"""TEST INFRASTRUCTURE ONLY — CPU restatement of the reference's noise schedule and DDIM sampler arithmetic.
Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference leg may import this.
Pinned by analytic known-answer values (SURVEY §8c) and against the unmodified reference sampler
(tests/test_oracle_cpu.py (test_*_matches_reference_golden*), tests/golden/).  Paths cited are relative to the reference
repository's root.
"""
from __future__ import annotations

import numpy as np
import torch


def linear_betas(n=1000, linear_start=0.00085, linear_end=0.012):
    """lvdm/models/utils_diffusion.py:31-35 ('linear' = linspace of sqrt(beta), squared, float64)."""
    return (torch.linspace(linear_start ** 0.5, linear_end ** 0.5, n, dtype=torch.float64) ** 2).numpy()


def zero_terminal_snr(betas):
    """utils_diffusion.py:112-144 (rescale_zero_terminal_snr)."""
    abar_sqrt = np.sqrt(np.cumprod(1.0 - betas, axis=0))
    a0, aT = abar_sqrt[0].copy(), abar_sqrt[-1].copy()
    abar_sqrt = (abar_sqrt - aT) * (a0 / (a0 - aT))
    abar = abar_sqrt ** 2
    alphas = np.concatenate([abar[0:1], abar[1:] / abar[:-1]])
    return 1.0 - alphas


def model_schedule(timesteps=1000, linear_start=0.00085, linear_end=0.012, zero_snr=True, base_scale=0.7,
                   turning_step=400):
    """ddpm3d.py:124-156 (register_schedule) + :523-528 (scale_arr).  Returns fp32 tensors like the buffers."""
    betas = linear_betas(timesteps, linear_start, linear_end)
    if zero_snr:
        betas = zero_terminal_snr(betas)
    ac = np.cumprod(1.0 - betas, axis=0)
    f32 = lambda a: torch.tensor(a, dtype=torch.float32)
    scale_arr = np.concatenate((np.linspace(1.0, base_scale, turning_step), np.full(timesteps, base_scale)))
    return dict(betas=f32(betas), alphas_cumprod=f32(ac), alphas_cumprod_prev=f32(np.append(1.0, ac[:-1])),
                sqrt_alphas_cumprod=f32(np.sqrt(ac)), sqrt_one_minus_alphas_cumprod=f32(np.sqrt(1.0 - ac)),
                scale_arr=f32(scale_arr))


def ddim_timesteps(S, n=1000, spacing="uniform_trailing"):
    """utils_diffusion.py:56-76."""
    if spacing == "uniform":
        return np.asarray(list(range(0, n, n // S))) + 1
    if spacing == "uniform_trailing":
        return np.flip(np.round(np.arange(n, 0, -(n / S)))).astype(np.int64) - 1
    raise NotImplementedError(spacing)


def ddim_tables(sched, S, eta, spacing="uniform_trailing"):
    """ddim.py:24-57 (make_schedule) + utils_diffusion.py:79-91: per-index alphas, alphas_prev, sigmas, scales.
    dtypes follow the reference: alphas fp32 tensor, alphas_prev float64 ndarray, sigmas float64 tensor."""
    ts = ddim_timesteps(S, sched["alphas_cumprod"].shape[0], spacing)
    ac = sched["alphas_cumprod"]
    alphas = ac[ts]
    alphas_prev = np.asarray([ac[0]] + ac[ts[:-1]].tolist())
    sigmas = eta * np.sqrt((1 - alphas_prev) / (1 - alphas) * (1 - alphas / alphas_prev))
    scale = sched["scale_arr"][ts]
    scale_prev = torch.cat([scale[0:1], scale[:-1]])
    return dict(timesteps=ts, alphas=alphas, alphas_prev=alphas_prev, sigmas=sigmas, scale=scale,
                scale_prev=scale_prev, sqrt_one_minus_alphas=np.sqrt(1.0 - alphas))


def step_coefficients(sched, tab, index):
    """The scalars p_sample_ddim materialises with torch.full(..., fp32) (ddim.py:251-254,263-264,271), in the
    reference's op order and precision.  Returns python floats (fp32-exact)."""
    t = int(tab["timesteps"][index])
    one = lambda v: torch.full((1,), float(v), dtype=torch.float32)
    a_prev = one(tab["alphas_prev"][index])
    sigma = one(tab["sigmas"][index])
    scale_t = one(tab["scale"][index])
    scale_prev = one(tab["scale_prev"][index])
    return dict(
        t=t,
        sqrt_ac=float(sched["sqrt_alphas_cumprod"][t]),
        sqrt_1mac=float(sched["sqrt_one_minus_alphas_cumprod"][t]),
        rescale=float(scale_prev / scale_t),
        sqrt_aprev=float(a_prev.sqrt()),
        dir_coef=float((1.0 - a_prev - sigma ** 2).sqrt()),
        sigma=float(sigma),
    )


def rescale_noise_cfg(noise_cfg, noise_pred_text, phi):
    """utils_diffusion.py:147-158."""
    dims = list(range(1, noise_cfg.ndim))
    std_text = noise_pred_text.std(dim=dims, keepdim=True)
    std_cfg = noise_cfg.std(dim=dims, keepdim=True)
    return phi * (noise_cfg * (std_text / std_cfg)) + (1 - phi) * noise_cfg


def ddim_update(x, e_c, e_uc, noise, co, cfg_scale, phi):
    """ddim.py:226-277 for the v-parameterisation with dynamic rescale (ddpm3d.py:240-252)."""
    v = e_uc + cfg_scale * (e_c - e_uc)          # in the dtype of the UNet outputs (fp16 under autocast, ddim.py:226)
    if phi > 0.0:
        v = rescale_noise_cfg(v, e_c, phi)
    v = v.float()                                 # the schedule buffers are fp32: buffer * v promotes (ddpm3d.py:240-252)
    eps = co["sqrt_ac"] * v + co["sqrt_1mac"] * x
    x0 = (co["sqrt_ac"] * x - co["sqrt_1mac"] * v) * co["rescale"]
    x_prev = co["sqrt_aprev"] * x0 + co["dir_coef"] * eps + co["sigma"] * noise
    return x_prev, x0


@torch.no_grad()
def sample(apply_model, sched, x_T, cond, uncond, S, eta=1.0, cfg_scale=7.5, phi=0.7, noises=None,
           spacing="uniform_trailing", fs=None, generator=None):
    """ddim.py:135-203 (ddim_sampling): apply_model(x, t, c, fs) -> v.  `noises[i]` (optional) is the N(0,1) draw
    of loop iteration i (teacher-forced tests); otherwise torch.randn with `generator`."""
    tab = ddim_tables(sched, S, eta, spacing)
    x = x_T
    B = x.shape[0]
    pred = None
    for i, step in enumerate(np.flip(tab["timesteps"])):
        index = S - i - 1
        ts = torch.full((B,), int(step), dtype=torch.long, device=x.device)
        e_c = apply_model(x, ts, cond, fs)
        e_uc = apply_model(x, ts, uncond, fs)
        nz = noises[i] if noises is not None else torch.randn(x.shape, generator=generator, device=x.device)
        x, pred = ddim_update(x, e_c, e_uc, nz, step_coefficients(sched, tab, index), cfg_scale, phi)
    return x, pred
