#!/usr/bin/env python
"""bench.py — ToonCrafter_512 hot path on B200: frames/sec at 320x512x16 frames, DDIM-50, CFG 7.5.

One "step" = one clip: DDIMSampler.sample (50 DDIM steps, cond + uncond UNet evaluation per step) followed by the
two dual-reference VAE decodes of scripts/evaluation/inference.py:262-270 (T = 16, then T = 14).  Weights are
seeded synthetic (no checkpoint / network here), inputs synthetic of the reference's shapes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--ddim-steps 50] [--impl reference]
                    [--config clip|decode|pair10] [--clips-per-step B] [--dump-outputs DIR]

--config clip   (default, BASELINE configs[1]/[2]/[4]) the step described above;
--config decode (configs[3]) step = the two decodes only;
--config pair10 (configs[0]) step = VAE-encode the reference's first 320x512 prompt pair (tests/golden fixture) +
                DDIM-10 + the two decodes — the configuration the CPU reference is quoted on.

--dump-outputs DIR writes the videos of the last timed step (rank 0's clips) as DIR/video_clip<c>.npy in float32.
The DDIM noise comes from torch's default generator, seeded before the warm-up, so runs with the same arguments see
the same inputs and noise and two builds can be compared output for output.

N > 1 is launched by torchrun (one process per GPU, shared-nothing clips, one NCCL weight broadcast at init).
Prints ONE JSON line (rank 0).  See DESIGN.md §Measurement for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

UNET_TF = 12.603                      # TFLOP per UNet forward per sample (SURVEY §8d, matmul/conv, 2 flops/MAC)
DEC_TF = {16: 37.875, 14: 33.148}     # TFLOP per decode pass
H, W, T = 40, 64, 16                  # latent geometry of 320x512, 16 frames


def clip_tflop(S):
    return 2 * S * UNET_TF + DEC_TF[16] + DEC_TF[14]


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return dict(tflops=float(d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0))), hbm=float(d["hbm_gbs"]),
                    src="measured (MEASURED_PEAKS.json, sustained cuBLAS bf16)")
    return dict(tflops=1400.0, hbm=6650.0, src="fallback (B200_PROFILING.md)")


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md recipe)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["nvidia-smi unavailable"])
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return dict(sm_mhz=sm[len(sm) // 2] if sm else None, sm_max_mhz=max(mx) if mx else None,
                    reasons=sorted(reasons), samples=len(sm))


# ---------------------------------------------------------------------------------------------------- model
def full_model_config():
    from tiny_config import FULL_DDCONFIG, FULL_UNET, model_config
    return model_config(FULL_UNET, FULL_DDCONFIG)


def build_model(dev, rank, world):
    """Full-size LatentVisualDiffusion with seeded synthetic weights; rank 0 generates, NCCL broadcasts."""
    from tooncrafter_b200 import diffusion, synthetic
    cfg = full_model_config()
    with torch.device("meta"):
        skeleton = diffusion.instantiate_from_config(cfg)
    m = skeleton.to_empty(device=dev)
    m.reset_schedule_buffers()
    with torch.no_grad():
        if rank == 0:
            for k, prm in m.named_parameters():
                prm.copy_(synthetic.synthetic_tensor(k, tuple(prm.shape), 0).to(dev))
        if world > 1:
            from tooncrafter_b200.distributed import broadcast_parameters
            # ONE broadcast of the weights at init (SURVEY §8e); no collective on the data path afterwards
            broadcast_parameters(m, src=0)
    m.perframe_ae = True
    return m.eval()


def host_inputs(seed):
    """Pinned host buffers of one clip's inputs (what scripts/evaluation/inference.py hands to the sampler)."""
    from tiny_config import FULL_DDCONFIG
    from tooncrafter_b200 import synthetic
    x_T, cond, uncond = synthetic.synthetic_inputs(1, T, H, W, 1024, seed=seed)
    ref = synthetic.synthetic_ref_context(FULL_DDCONFIG["ch"], FULL_DDCONFIG["ch_mult"], 8 * H, 8 * W, seed=seed)
    pin = lambda t: t.contiguous().pin_memory()
    return dict(x_T=pin(x_T), ctx_c=pin(cond["c_crossattn"][0]), ctx_u=pin(uncond["c_crossattn"][0]),
                c_concat=pin(cond["c_concat"][0]), ref=[pin(r.half()) for r in ref])


def to_device(hi, dev):
    cc = hi["c_concat"].to(dev, non_blocking=True)
    d = dict(x_T=hi["x_T"].to(dev, non_blocking=True),
             cond={"c_crossattn": [hi["ctx_c"].to(dev, non_blocking=True)], "c_concat": [cc]},
             uncond={"c_crossattn": [hi["ctx_u"].to(dev, non_blocking=True)], "c_concat": [cc]},
             ref=[r.to(dev, non_blocking=True) for r in hi["ref"]])
    return d


def h2d_bytes(hi):
    n = sum(hi[k].numel() * hi[k].element_size() for k in ("x_T", "ctx_c", "ctx_u", "c_concat"))
    return n + sum(r.numel() * r.element_size() for r in hi["ref"])


def run_clip(model, sampler, di, S, fs):
    """The hot path through the reference-facing API: sample() + the two decode_first_stage() calls."""
    samples, _ = sampler.sample(S=S, batch_size=1, shape=[4, T, H, W], conditioning=di["cond"],
                                unconditional_conditioning=di["uncond"], eta=1.0, unconditional_guidance_scale=7.5,
                                x_T=di["x_T"], fs=fs, timestep_spacing="uniform_trailing", guidance_rescale=0.7,
                                verbose=False)
    trimmed = torch.cat([samples[:, :, :1], samples[:, :, 2:-2], samples[:, :, -1:]], dim=2)   # drop frames 1 and 14
    group = getattr(sampler, "latency_group", None)
    if group is None:
        video = model.decode_first_stage(samples, ref_context=di["ref"])
        video2 = model.decode_first_stage(trimmed, ref_context=di["ref"])
        video[:, :, 7:9] = video2[:, :, 6:8]                                                    # inference.py:264-270
        return video
    # latency mode: both ranks hold identical samples; pair-rank 0 decodes the 16 frames, pair-rank 1 the 14-frame
    # variant at the same time and ships its two middle frames over
    import torch.distributed as dist
    r = dist.get_rank(group)
    if r == 0:
        video = model.decode_first_stage(samples, ref_context=di["ref"])
        patch = torch.empty_like(video[:, :, 7:9]).contiguous()
    else:
        video = model.decode_first_stage(trimmed, ref_context=di["ref"])
        patch = video[:, :, 6:8].contiguous()
    dist.broadcast(patch, src=dist.get_global_rank(group, 1), group=group)
    if r == 0:
        video[:, :, 7:9] = patch
    return video


def workload_config(S, config="clip", clips_per_step=1):
    """The `config` object of the JSON line (both arms name the same workload, key for key)."""
    return {"config": config, "clips_per_gpu_per_step": clips_per_step, "workload": "ToonCrafter_512 320x512x16f DDIM-%d fp16, CFG 7.5 (cond+uncond batched), eta 1.0, "
                        "uniform_trailing, guidance_rescale 0.7, sample() + decode T=16 + decode T=14; "
                        "1 clip per GPU per step; random-init weights, synthetic inputs" % S,
            "l2": "working set per clip (2.9 GB fp16 weights + activations) exceeds the 126 MB L2",
            "baseline_note": "vs_baseline = value / 0.667 frames/s (README.md:222: ~24 s/clip on A100)"}


# ---------------------------------------------------------------------------------------------------- roofline
def gemm_roofline(model, dev):
    """Live per-launch CUDA-event timing of every tc_gemm_kernel launch of one eager UNet forward (B = 2)."""
    from tooncrafter_b200 import ops
    eng = model.model.diffusion_model._engine
    plan = eng.plan_for(2, T, H, W, 77 + 16 * T)
    stream = torch.cuda.current_stream()
    recs = []
    for fn, a, kw in plan.main.calls:
        if fn is ops.conv_gemm:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn(*a, **kw)
            e1.record(stream)
            a_dims, taps, out_dims, n_cols = a[1], a[4], a[6], a[7]
            M = out_dims[0] * out_dims[1] * out_dims[2]
            fl = 2.0 * M * n_cols * len(taps) * a_dims[3]
            recs.append((e0, e1, fl, (M, n_cols, a_dims[3], len(taps), tuple(out_dims))))
        else:
            fn(*a, **kw)
    torch.cuda.synchronize()
    tot_ms = sum(e0.elapsed_time(e1) for e0, e1, _, _ in recs)
    tot_fl = sum(fl for _, _, fl, _ in recs)
    shapes = {}
    for e0, e1, fl, key in recs:
        d = shapes.setdefault(key, dict(n=0, ms=0.0, flops=fl))
        d["n"] += 1
        d["ms"] += e0.elapsed_time(e1)
    return dict(launches=len(recs), avg_launch_us=1e3 * tot_ms / max(len(recs), 1), tflops=tot_fl / tot_ms / 1e9,
                flops_per_launch=tot_fl / max(len(recs), 1), gemm_ms_per_forward=tot_ms, shapes=shapes)


# ---------------------------------------------------------------------------------------------------- CPU arm
def gemm_traffic():
    """(dram bytes per tc_gemm_kernel launch, provenance) from the committed ncu launch list, or (None, reason)."""
    prof = Path(__file__).resolve().parent / "profiles"
    p = prof / "r02_unet_b2_launches.gemm_traffic.json"
    if not p.exists():
        p = prof / "r01_unet_b2_launches_final.gemm_traffic.json"
    try:
        d = json.loads(p.read_text())
        return float(d["dram_bytes_per_launch"]), f"profiles/{p.name}: {d['launches']} launches, {d['source']}"
    except Exception as e:      # noqa: BLE001 - the file is optional evidence, not a dependency of the measurement
        return None, f"no ncu capture committed ({type(e).__name__})"


def cpu_threads():
    """Host threads for the CPU arm: all cores up to 32 (beyond that the fp32 conv/GEMM mix of this UNet stops
    scaling and oversubscribed boxes get slower: 128 threads measured 185 s/forward vs 35 s on 8 dedicated cores)."""
    return max(1, min(os.cpu_count() or 1, 32))


CPU_ARM_CACHE = Path(tempfile.gettempdir()) / "tooncrafter_b200_cpu_reference_arm.json"   # not in the tree: it may be read-only


def reference_source():
    """Which implementation the CPU arm executes.  The reference is pure Python without setup.py / pyproject.toml, so
    `pip install --target baseline/_ref /root/reference` fails ("not installable", DESIGN.md §5) and /root/reference does
    not exist on the GPU box: unless someone placed an importable copy under baseline/_ref (looked for here), the arm
    runs the oracle port — the same algorithm, pinned to the reference by the committed goldens."""
    ref = ROOT / "baseline" / "_ref"
    if (ref / "lvdm" / "models" / "ddpm3d.py").exists():
        return "reference", str(ref)
    return "port", "baseline/_ref absent (reference not pip-installable); oracle/ port of the same algorithm"


class CpuReference:
    """The reference algorithm on the host cores (fp32, all threads): full-size seeded synthetic weights built once,
    then timed samples: one UNet forward (B = 1) and one T = 16 decode."""

    def __init__(self, threads):
        from tiny_config import FULL_DDCONFIG, FULL_UNET
        from tooncrafter_b200 import diffusion, layout, modules, synthetic
        torch.set_num_threads(threads)
        self.kind, self.why = reference_source()
        self.ulay = layout.unet_layout(FULL_UNET)
        self.dlay = layout.decoder_layout(FULL_DDCONFIG)
        t0 = time.perf_counter()
        with torch.device("meta"):
            sk = modules.UNetModel(**FULL_UNET)
            ae = diffusion.AutoencoderKL_Dualref(ddconfig=FULL_DDCONFIG, embed_dim=4)
        self.sd = {}
        for k, p in sk.named_parameters():
            key = "model.diffusion_model." + k
            self.sd[key] = synthetic.synthetic_tensor(key, tuple(p.shape), 0)
        for k, p in ae.decoder.named_parameters():
            key = "first_stage_model.decoder." + k
            self.sd[key] = synthetic.synthetic_tensor(key, tuple(p.shape), 0)
        self.build_s = time.perf_counter() - t0
        x_T, cond, _ = synthetic.synthetic_inputs(1, T, H, W, 1024, seed=123)
        self.xc = torch.cat([x_T] + cond["c_concat"], 1)
        self.ctx = cond["c_crossattn"][0]
        self.z = x_T * 0.18215 * 3
        self.ref = synthetic.synthetic_ref_context(FULL_DDCONFIG["ch"], FULL_DDCONFIG["ch_mult"], 8 * H, 8 * W, seed=123)

    def unet_forward_seconds(self):
        from oracle import unet_oracle
        t0 = time.perf_counter()
        unet_oracle.unet_forward(self.sd, self.ulay, self.xc, torch.tensor([500]), self.ctx, torch.tensor([10]),
                                 "model.diffusion_model.")
        return time.perf_counter() - t0

    def decode16_seconds(self):
        from oracle import vae_oracle
        t0 = time.perf_counter()
        vae_oracle.decode_first_stage(self.sd, self.dlay, self.z, self.ref, chunk=16)
        return time.perf_counter() - t0


def cpu_sec_per_clip(t_fwd, t_dec16, S):
    """2*S UNet forwards (measured) + decode T=16 (measured) + decode T=14 (the T=16 time scaled by its flops)."""
    return 2 * S * t_fwd + t_dec16 * (1.0 + DEC_TF[14] / DEC_TF[16])


def reference_arm(args):
    """--impl reference: the reference algorithm on the box's host cores.  Each timed step is a bounded sample = ONE
    full-size UNet forward (B = 1, 12.6 TFLOP); before the steps ONE T = 16 decode (37.9 TFLOP) is timed as well.
    sec/clip = 2*S*forward + decodes with every term measured on this box (the T = 14 decode is the T = 16 time
    scaled by flops)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = cpu_threads()
    S = args.ddim_steps
    ref = CpuReference(cores)
    t_dec = ref.decode16_seconds()
    times = []
    for i in range(args.warmup + args.steps):
        dt = ref.unet_forward_seconds()
        if i >= args.warmup:
            times.append(dt)
    t_fwd = sum(times) / len(times)
    sec_per_clip = cpu_sec_per_clip(t_fwd, t_dec, S)
    fps = 16.0 / sec_per_clip
    sample = (f"{len(times)} x one full-size UNet forward (B=1, fp32) = {t_fwd:.1f} s each + one T=16 decode = {t_dec:.1f} s, "
              f"seeded synthetic weights ({ref.build_s:.0f} s to build), {cores} threads; sec/clip = {2 * S} forwards + "
              f"decode16 + decode14 (decode16 x {DEC_TF[14] / DEC_TF[16]:.3f}) = {sec_per_clip:.0f} s; {ref.why}")
    cb = {"value": fps, "unit": "frames/s", "cores": cores, "kind": ref.kind, "sample": sample,
          "unet_forward_s": t_fwd, "decode16_s": t_dec, "sec_per_clip": sec_per_clip}
    out = {"impl": "reference", "metric": "frames/sec (320x512x16f, DDIM-%d)" % S, "value": fps, "unit": "frames/s",
           "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_fwd,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": workload_config(S, args.config, args.clips_per_step), "cpu_baseline": cb,
           "e2e": {"value": fps, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    try:
        CPU_ARM_CACHE.write_text(json.dumps(dict(cb, when=time.time(), ddim_steps=S)))
    except OSError:
        pass
    print(json.dumps(out), flush=True)
    return 0


def cpu_baseline_for_main_arm(S):
    """cpu_baseline of the B200 line: the reference arm's measurement when it ran on THIS box within the last hour (the
    driver runs it immediately before), otherwise one fresh bounded sample (one UNet forward + one decode)."""
    try:
        d = json.loads(CPU_ARM_CACHE.read_text())
        if time.time() - d["when"] < 3600 and d["ddim_steps"] == S:
            d.pop("when")
            d.pop("ddim_steps")
            d["sample"] = "reused from `bench.py --impl reference` on this box minutes earlier: " + d["sample"]
            return d
    except (OSError, KeyError, ValueError):
        pass
    cores = cpu_threads()
    ref = CpuReference(cores)
    t_fwd = ref.unet_forward_seconds()                      # bounded sample: ~25 s of CPU work
    t_dec = t_fwd * DEC_TF[16] / UNET_TF                    # the decode is NOT run here (it alone is > 1 min of CPU)
    spc = cpu_sec_per_clip(t_fwd, t_dec, S)
    return {"value": 16.0 / spc, "unit": "frames/s", "cores": cores, "kind": ref.kind, "unet_forward_s": t_fwd,
            "decode16_s": None, "sec_per_clip": spc,
            "sample": f"one full-size UNet forward (B=1, fp32) = {t_fwd:.1f} s on {cores} threads, seeded synthetic weights; "
                      f"sec/clip = {2 * S} forwards + decodes scaled by flops from the forward (`bench.py --impl reference` "
                      f"measures the decode too and this field reuses it when it ran on the same box); {ref.why}"}


# ---------------------------------------------------------------------------------------------------- library arm
def library_baseline(model, di, fs, S, roof):
    """The reference ALGORITHM on this same GPU through stock PyTorch kernels (cuDNN conv, cuBLAS GEMM, SDPA flash
    attention) under torch.autocast(fp16) with fp32 parameters — what scripts/evaluation/inference.py:323 executes with
    xformers installed.  This is the number a user gets for free from PyTorch on a B200, i.e. the one to beat.
    One DDIM step = two B = 1 UNet forwards (ddim.py:221-222); plus the T = 16 and T = 14 decodes."""
    from oracle import unet_oracle, vae_oracle
    from tiny_config import FULL_DDCONFIG, FULL_UNET
    from tooncrafter_b200 import layout
    sd = model.state_dict()
    ulay, dlay = layout.unet_layout(FULL_UNET), layout.decoder_layout(FULL_DDCONFIG)
    x = di["x_T"]
    ts = torch.full((1,), 500, device=x.device, dtype=torch.long)
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def unet_step():
        for c in (di["cond"], di["uncond"]):
            xc = torch.cat([x] + c["c_concat"], 1)
            unet_oracle.unet_forward(sd, ulay, xc, ts, torch.cat(c["c_crossattn"], 1), fs, "model.diffusion_model.")

    def decodes():
        ref = [r.float() for r in di["ref"]]
        z = x * 0.18215 * 3
        vae_oracle.decode_first_stage(sd, dlay, z, ref, chunk=16)
        vae_oracle.decode_first_stage(sd, dlay, torch.cat([z[:, :, :1], z[:, :, 2:-2], z[:, :, -1:]], 2), ref, chunk=14)

    def timed(fn, reps):
        with torch.autocast("cuda", dtype=torch.float16), torch.no_grad():
            fn()
            torch.cuda.synchronize()
            e0, e1 = ev(), ev()
            e0.record()
            for _ in range(reps):
                fn()
            e1.record()
            torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    out = {}
    for impl in ("sdpa", "einsum"):
        unet_oracle.ATTENTION_IMPL = impl
        try:
            out[f"unet_step_ms_{impl}"] = timed(unet_step, 3)
        except torch.cuda.OutOfMemoryError:
            out[f"unet_step_ms_{impl}"] = None
    unet_oracle.ATTENTION_IMPL = "einsum"
    out["decodes_ms"] = timed(decodes, 2)
    best = min(v for k, v in out.items() if k.startswith("unet_step_ms") and v)
    spc = (S * best + out["decodes_ms"]) / 1e3
    out.update(sec_per_clip=spc, frames_per_s=16.0 / spc, tflops=clip_tflop(S) / spc,
               what="reference algorithm (oracle walk over the same fp32 weights) under torch.autocast(fp16) on this GPU: "
                    "cuDNN / cuBLAS / SDPA; eager PyTorch, no CUDA graph; sec/clip = S x (two B=1 forwards) + both decodes")
    # per-shape: the ten GEMM shapes that cost this framework the most, against cuBLAS / cuDNN on the same shape
    top = sorted(roof["shapes"].items(), key=lambda kv: -kv[1]["ms"])[:10]
    rows = []
    for (M, N, K, taps, odims), d in top:
        ours_us = 1e3 * d["ms"] / d["n"]
        if taps == 1:
            a = torch.randn(M, K, device=x.device, dtype=torch.float16)
            w = torch.randn(N, K, device=x.device, dtype=torch.float16)
            fn = lambda: torch.matmul(a, w.t())
            lib = "cuBLAS fp16 matmul"
        elif taps == 9:
            n_, h_, w_ = odims
            a = torch.randn(n_, K, h_, w_, device=x.device, dtype=torch.float16).to(memory_format=torch.channels_last)
            w = torch.randn(N, K, 3, 3, device=x.device, dtype=torch.float16).to(memory_format=torch.channels_last)
            fn = lambda: torch.nn.functional.conv2d(a, w, padding=1)
            lib = "cuDNN fp16 conv3x3 (channels_last; stride-1 stand-in)"
        else:
            b_, t_, hw_ = odims
            a = torch.randn(b_, K, t_, hw_, 1, device=x.device, dtype=torch.float16)
            w = torch.randn(N, K, 3, 1, 1, device=x.device, dtype=torch.float16)
            fn = lambda: torch.nn.functional.conv3d(a, w, padding=(1, 0, 0))
            lib = "cuDNN fp16 conv3d (3,1,1)"
        try:
            with torch.no_grad():
                for _ in range(3):
                    fn()
                e0, e1 = ev(), ev()
                e0.record()
                for _ in range(10):
                    fn()
                e1.record()
                torch.cuda.synchronize()
            lib_us = 1e3 * e0.elapsed_time(e1) / 10
        except RuntimeError:
            lib_us = None
        rows.append(dict(M=M, N=N, K=K, taps=taps, launches_per_forward=d["n"], ours_us=round(ours_us, 1),
                         library_us=None if lib_us is None else round(lib_us, 1), library=lib,
                         ours_tflops=round(d["flops"] / ours_us / 1e6, 1)))
    out["gemm_shapes_top10"] = rows
    return out


# ---------------------------------------------------------------------------------------------------- main
def pair_inputs(model, dev, S):
    """BASELINE config #1 inputs: the reference's first 512_interp prompt pair (tests/golden/prompt_pair_74906.npz, made
    by tests/golden/make_prompt_pair.py with the transform of inference.py:65-69) as a pinned uint8 host buffer."""
    import numpy as np
    f = np.load(ROOT / "tests" / "golden" / "prompt_pair_74906.npz")["frames"]          # [2, 320, 512, 3] uint8
    return torch.from_numpy(f).pin_memory()


def run_pair(model, sampler, frames_u8_host, di, S, fs, dev):
    """Config #1 through the public API: frames -> first_stage_model.encode(return_hidden_states=True) -> c_concat and
    ref_context (inference.py:164-200) -> sample(S) -> both decodes.  Only the two DISTINCT frames are encoded (the
    reference encodes 8 copies of each, SURVEY 8f-1); text / image embeddings are synthetic (no CLIP weights here)."""
    fr = frames_u8_host.to(dev, non_blocking=True).permute(0, 3, 1, 2).float() / 127.5 - 1.0      # [2, 3, 320, 512]
    post, hidden = model.first_stage_model.encode(fr, return_hidden_states=True)
    z2 = model.get_first_stage_encoding(post)                                                     # [2, 4, 40, 64]
    cc = torch.zeros(1, 4, T, H, W, device=dev)
    cc[0, :, 0], cc[0, :, -1] = z2[0], z2[1]
    ref = [h.reshape(1, 2, *h.shape[1:]).permute(0, 2, 1, 3, 4).contiguous() for h in hidden]
    dj = dict(x_T=di["x_T"], ref=ref,
              cond={"c_crossattn": di["cond"]["c_crossattn"], "c_concat": [cc]},
              uncond={"c_crossattn": di["uncond"]["c_crossattn"], "c_concat": [cc]})
    return run_clip(model, sampler, dj, S, fs)


def run_decode(model, z, ref):
    """Config #4: the two decode_first_stage passes of inference.py:262-270 on given latents."""
    video = model.decode_first_stage(z, ref_context=ref)
    trimmed = torch.cat([z[:, :, :1], z[:, :, 2:-2], z[:, :, -1:]], dim=2)
    video2 = model.decode_first_stage(trimmed, ref_context=ref)
    video[:, :, 7:9] = video2[:, :, 6:8]
    return video


DUMP_BUDGET_BYTES = 60_000_000      # data bytes: with the .npy headers the files stay under 64 MB


def dump_outputs(out_dir, arrays):
    """Write {name: float32 host tensor} as out_dir/<name>.npy.  Past DUMP_BUDGET_BYTES in all, each array is replaced by
    a fixed sample of its flattened elements (positions from numpy's default_rng(0), sorted), the same in every run."""
    import numpy as np
    out_dir = Path(out_dir)
    out_dir.mkdir(parents=True, exist_ok=True)
    total = sum(a.numel() for a in arrays.values()) * 4
    for name, t in arrays.items():
        a = t.numpy()
        if total > DUMP_BUDGET_BYTES:
            a = a.reshape(-1)
            k = a.size * DUMP_BUDGET_BYTES // total
            a = a[np.sort(np.random.default_rng(0).choice(a.size, size=k, replace=False))]
        np.save(out_dir / f"{name}.npy", a.astype(np.float32, copy=False))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--ddim-steps", type=int, default=None, help="default 50 (10 for --config pair10)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="clip", choices=["clip", "decode", "pair10"],
                    help="clip: sample() + both decodes (BASELINE configs 2/3/5); decode: both decodes only (config 4); "
                         "pair10: encode the reference's prompt pair + DDIM-10 + decodes (config 1)")
    ap.add_argument("--clips-per-step", type=int, default=1,
                    help="B independent clips per GPU per step, run back to back (B > 1 = B independent B = 1 runs, "
                         "SURVEY 8e: the reference's decoder is only defined for one clip per call)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library-baseline", action="store_true")
    ap.add_argument("--latency-mode", action="store_true",
                    help="pairs of GPUs share one clip: each evaluates one classifier-free-guidance branch per step "
                         "(one NCCL all-gather per step) and one of the two decodes; needs an even --gpus >= 2")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the videos of the last timed step as DIR/video_clip<c>.npy (float32, at most 64 MB)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.ddim_steps is None:
        args.ddim_steps = 10 if args.config == "pair10" else 50
    if args.impl == "reference":
        return reference_arm(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    from tooncrafter_b200 import ops
    from tooncrafter_b200.sampler import DDIMSampler
    S = args.ddim_steps
    Bc = args.clips_per_step
    model = build_model(dev, rank, world)
    sampler = DDIMSampler(model)
    fs = torch.tensor([10], device=dev)
    from tooncrafter_b200.distributed import clip_seed, shard_clips
    pair_group, in_pair = None, 0
    if args.latency_mode:
        if world < 2:
            raise SystemExit("--latency-mode needs torchrun with an even number of GPUs >= 2")
        from tooncrafter_b200.distributed import latency_pairs
        pair_group, my_clip, in_pair = latency_pairs()     # one clip per GPU PAIR per step
        sampler.latency_group = pair_group
        my_clips = [my_clip]
    else:
        my_clips = shard_clips(world * Bc, rank, world)    # Bc clips per GPU per step (weak scaling)
    # per-clip seed: results independent of the world size
    his = [host_inputs(seed=clip_seed(123, c)) for c in my_clips]
    dis = [to_device(hi, dev) for hi in his]
    hi, di = his[0], dis[0]
    frames_host = pair_inputs(model, dev, S) if args.config == "pair10" else None
    torch.cuda.synchronize()

    def one_step(inputs):
        """One step of the selected config on device-resident `inputs` (list of per-clip dicts); returns the videos."""
        vs = []
        for dj in inputs:
            if args.config == "clip":
                vs.append(run_clip(model, sampler, dj, S, fs))
            elif args.config == "decode":
                vs.append(run_decode(model, dj["z"], dj["ref"]))
            else:
                vs.append(run_pair(model, sampler, frames_host, dj, S, fs, dev))
        return vs

    if args.config == "decode":
        for hj, dj in zip(his, dis):
            hj["z"] = (hj["x_T"] * 0.18215 * 3).pin_memory()
            dj["z"] = hj["z"].to(dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    torch.manual_seed(0)            # the DDIM noise (eta = 1): same arguments, same outputs
    # ---- warm-up (builds plans, captures graphs) ------------------------------------------------------------
    for _ in range(max(args.warmup, 1)):
        one_step(dis)
    barrier()

    # ---- timed: device-resident inputs ----------------------------------------------------------------------
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for _ in range(args.steps):
        videos = one_step(dis)
    e1.record()
    barrier()
    ms_dev = max_over_ranks(e0.elapsed_time(e1))
    clk = clocks.stop() if rank == 0 else None
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = {f"video_clip{c}": v.float().cpu() for c, v in zip(my_clips, videos)}

    # ---- timed: end to end through the public API with HOST buffers -----------------------------------------
    out_host = torch.empty(1, 3, T, 8 * H, 8 * W, dtype=torch.float16).pin_memory()

    def step_h2d(hj):
        if args.config == "decode":
            return dict(z=hj["z"].to(dev, non_blocking=True), ref=[r.to(dev, non_blocking=True) for r in hj["ref"]])
        return to_device(hj, dev)

    def step_h2d_bytes(hj):
        if args.config == "decode":
            return hj["z"].numel() * 4 + sum(r.numel() * r.element_size() for r in hj["ref"])
        if args.config == "pair10":       # frames + synthetic embeddings + x_T (ref_context comes from the encoder)
            return frames_host.numel() + sum(hj[k].numel() * hj[k].element_size() for k in ("x_T", "ctx_c", "ctx_u", "c_concat"))
        return h2d_bytes(hj)

    barrier()
    e0.record()
    for _ in range(args.steps):
        for hj in his:
            dj = step_h2d(hj)                              # H2D of this clip's inputs from pinned memory
            video = one_step([dj])[0]
            out_host[:, :, :video.shape[2]].copy_(video, non_blocking=True)   # D2H of the clip (latency mode: pair-rank 1
                                                                              # holds the 14-frame variant)
    e1.record()
    barrier()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    peaks = load_peaks()
    unet = model.model.diffusion_model
    dec = model.first_stage_model._dec_engine
    # launches inside captured graphs are replayed, not re-issued through the C ABI: count them from the programs
    kernels_unet, roof = 0, None
    if args.config != "decode":
        plan = unet._engine.plan_for(2, T, H, W, 77 + 16 * T)
        roof = gemm_roofline(model, dev)
        c0 = ops.launch_count()
        plan.main.run()
        torch.cuda.synchronize()
        kernels_unet = ops.launch_count() - c0
        plan.ctx.run()
        torch.cuda.synchronize()
        kernels_ctx = ops.launch_count() - c0 - kernels_unet
    kernels_dec = 0
    for key in ((16, H, W), (14, H, W)):
        pl = dec.plan_for(*key)
        c0 = ops.launch_count()
        pl.main.run()
        pl.ctx.run()
        torch.cuda.synchronize()
        kernels_dec += ops.launch_count() - c0
    launches_per_clip = kernels_dec + (S * (kernels_unet + 2) + kernels_ctx if args.config != "decode" else 0)
    clips = args.steps * Bc * (world // 2 if args.latency_mode else world)
    fps_dev = 16.0 * clips / (ms_dev / 1e3)
    fps_e2e = 16.0 * clips / (ms_e2e / 1e3)
    tf_clip = clip_tflop(S) if args.config != "decode" else DEC_TF[16] + DEC_TF[14]
    metric = {"clip": "frames/sec (320x512x16f, DDIM-%d)" % S,
              "decode": "frames/sec (dual-reference VAE decode only, 320x512x16f, T=16 + T=14 passes)",
              "pair10": "frames/sec (320x512x16f, DDIM-%d, encode + sample + decode of the 512_interp prompt pair)" % S}[args.config]
    cfg = workload_config(S, args.config, Bc)
    if args.config == "decode":
        cfg["workload"] = ("ToonCrafter_512 AutoencoderKL_Dualref decode only: 16 latents 40x64 -> 320x512x16f (T=16 pass + "
                           "T=14 pass, inference.py:262-270) fp16; random-init weights, synthetic latents / reference maps")
    elif args.config == "pair10":
        cfg["workload"] = ("ToonCrafter_512 320x512x16f on prompts/512_interp/74906_1462_frame{1,3}.png (fixture), VAE encode "
                           "with hidden states + DDIM-%d CFG 7.5 + decode T=16 + decode T=14, fp16; random-init weights, "
                           "synthetic text/image embeddings" % S)
    per_step_ms = ms_dev / args.steps
    out = {
        "metric": metric, "value": fps_dev, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step_ms, "higher_is_better": True,
        "scaling": "strong" if args.latency_mode else "weak",
        "vs_baseline": fps_dev / (16.0 / 24.0) if (S == 50 and args.config == "clip") else None, "dtype": "f16",
        "data": "synthetic",
        "config": cfg,
        "sec_per_clip": per_step_ms / Bc / 1e3,
        "mode": "latency (one clip per GPU pair: CFG branches split, all-gather per step)" if args.latency_mode
                else "throughput (%d clip(s) per GPU per step)" % Bc,
        "tflops_per_gpu": tf_clip * Bc / (per_step_ms / 1e3) / (2 if args.latency_mode else 1),
        "e2e": {"value": fps_e2e, "unit": "frames/s", "h2d_bytes_per_step": sum(step_h2d_bytes(hj) for hj in his),
                "d2h_bytes_per_step": Bc * out_host.numel() * out_host.element_size(),
                "sec_per_clip": ms_e2e / args.steps / Bc / 1e3},
        "gpu_launches": launches_per_clip * args.steps * Bc,
        "timed_region_note": "the per-conditioning context K/V program and the reference-map packing program run on every "
                             "sample() / decode() call, inside both timed regions",
        "clocks": clk,
    }
    if roof is not None:
        out["roofline"] = {"bound": "tensor", "kernel": "tc_gemm_kernel (implicit-GEMM conv / linear, tcgen05)",
                           "achieved": roof["tflops"], "peak": peaks["tflops"], "unit": "TFLOP/s",
                           "frac": roof["tflops"] / peaks["tflops"], "traffic": gemm_traffic()[0],
                           "traffic_unit": "bytes of DRAM read+write per launch (ncu, average over the GEMM launches of one UNet forward)",
                           "traffic_source": gemm_traffic()[1], "peak_source": peaks["src"],
                           "launches_per_unet_forward": roof["launches"], "avg_launch_us": roof["avg_launch_us"],
                           "flops_per_launch": roof["flops_per_launch"],
                           "share_of_unet_forward": roof["gemm_ms_per_forward"]}
    if world == 1 and args.config == "clip" and not args.no_library_baseline:
        try:
            out["library_baseline"] = library_baseline(model, di, fs, S, roof)
        except Exception as e:       # noqa: BLE001 - an optional comparison must not lose the measured line
            out["library_baseline"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    if not args.no_cpu_baseline and world == 1:
        out["cpu_baseline"] = cpu_baseline_for_main_arm(S)
    print(json.dumps(out), flush=True)
    if dumped is not None:
        dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
