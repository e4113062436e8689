"""Shared by tests/golden/make_golden_glue.py (drives the UNMODIFIED reference with its own glue function
scripts/evaluation/funcs.py::batch_ddim_sampling, :14-93) and tests/glue_driver.py (drives this repository's alias
tree with `batch_ddim_sampling` below, which makes the same calls) on the tiny configuration.

Conditioning stages (CLIP text / image towers, Resampler) are outside the hot path: both sides install the same seeded
test doubles for `get_learned_conditioning`, `embedder` and `image_proj_model`."""
import torch

SEED_RNG = 77
STEPS = 4


def batch_ddim_sampling(model, cond, noise_shape, n_samples=1, ddim_steps=50, ddim_eta=1.0, cfg_scale=1.0, hs=None,
                        temporal_cfg_scale=None, **kwargs):
    """What the reference's inference scripts do around the model (funcs.py:14-93), for the case they run: an
    "empty_seq" unconditional branch with a zero image token, DDIMSampler.sample with the scripts' keyword set
    (clean_cond, temporal_length, conditional_guidance_scale_temporal, timestep spacing and guidance rescale chosen by
    the latent width), then two dual-reference decodes, the second without frames 1 and T-2, whose two middle frames
    replace the first decode's.  Returns [B, n_samples, C, T, H, W]."""
    from lvdm.models.samplers.ddim import DDIMSampler            # the alias, as the scripts import it
    sampler = DDIMSampler(model)
    B, T = noise_shape[0], noise_shape[2]
    fs = cond.pop("fs")
    spacing, rescale = ("uniform", 0.0) if noise_shape[-1] == 32 else ("uniform_trailing", 0.7)
    assert cfg_scale != 1.0 and model.uncond_type == "empty_seq"
    uc_img = model.image_proj_model(model.embedder(torch.zeros(B, 3, 224, 224).to(model.device)))
    uc = dict(cond, c_crossattn=[torch.cat([model.get_learned_conditioning(B * [""]), uc_img], dim=1)])
    variants = []
    for _ in range(n_samples):
        samples, _ = sampler.sample(S=ddim_steps, conditioning=cond, batch_size=B, shape=noise_shape[1:], verbose=False,
                                    unconditional_guidance_scale=cfg_scale, unconditional_conditioning=uc, eta=ddim_eta,
                                    temporal_length=T, conditional_guidance_scale_temporal=temporal_cfg_scale,
                                    x_T=None, fs=fs, timestep_spacing=spacing, guidance_rescale=rescale,
                                    **dict(kwargs, clean_cond=True))
        video = model.decode_first_stage(samples, ref_context=hs)
        keep = [i for i in range(T) if i not in (1, T - 2)]
        middle = model.decode_first_stage(samples[:, :, keep], ref_context=hs)
        Tv = video.shape[2]
        video[:, :, Tv // 2 - 1:Tv // 2 + 1] = middle[:, :, Tv // 2 - 2:Tv // 2]
        variants.append(video)
    return torch.stack(variants, dim=1)


class _Fn(torch.nn.Module):
    """A parameter-free nn.Module around a callable (the conditioning stages are registered sub-modules)."""

    def __init__(self, fn):
        super().__init__()
        self._fn = fn

    def forward(self, *a, **k):
        return self._fn(*a, **k)


def install_conditioning_doubles(model, T, ctx_dim):
    from tooncrafter_b200 import synthetic
    g = lambda n: synthetic._gen(n, 555)
    txt_empty = torch.randn(1, 77, ctx_dim, generator=g("glue.txt.empty"))
    img_zero = torch.randn(1, 16 * T, ctx_dim, generator=g("glue.img.zero"))
    model.get_learned_conditioning = lambda prompts: txt_empty.expand(len(prompts), -1, -1).clone()
    model.embedder = _Fn(lambda img: img.new_zeros(img.shape[0], 4, ctx_dim))
    model.image_proj_model = _Fn(lambda tok: img_zero.expand(tok.shape[0], -1, -1).clone())


def glue_inputs(T, h, w, ctx_dim):
    from tooncrafter_b200 import synthetic
    g = lambda n: synthetic._gen(n, 556)
    frames = torch.rand(2, 3, 8 * h, 8 * w, generator=g("glue.frames")) * 2 - 1
    z = torch.randn(1, 4, T, h, w, generator=g("glue.z")) * 0.18215 * 3
    cc = torch.zeros_like(z)
    cc[:, :, 0], cc[:, :, -1] = z[:, :, 0], z[:, :, -1]
    prompts = [torch.randn(1, 77 + 16 * T, ctx_dim, generator=g(f"glue.ctx.{i}")) for i in range(2)]
    mask = (torch.rand(1, 1, T, h, w, generator=g("glue.mask")) > 0.5).float()
    x0 = torch.randn(1, 4, T, h, w, generator=g("glue.x0"))
    return dict(frames=frames, c_concat=cc, prompts=prompts, mask=mask, x0=x0, fs=torch.tensor([10]))


def run_glue(batch_ddim_sampling, model, T, h, w, ctx_dim):
    """Two prompts back to back (a stale conditioning cache would show in the second), then prompt 0 again with the
    mask / x0 blending kwargs (ddim.py:174-180).  Returns the three decoded clips."""
    gi = glue_inputs(T, h, w, ctx_dim)
    install_conditioning_doubles(model, T, ctx_dim)
    with torch.no_grad():
        post, hidden = model.first_stage_model.encode(gi["frames"], return_hidden_states=True)
        hs = [hh.reshape(1, 2, *hh.shape[1:]).permute(0, 2, 1, 3, 4).contiguous().float() for hh in hidden]
        outs = []
        for k, extra in ((0, {}), (1, {}), (0, dict(mask=gi["mask"], x0=gi["x0"]))):
            cond = {"c_crossattn": [gi["prompts"][k].clone()], "c_concat": [gi["c_concat"]], "fs": gi["fs"]}
            torch.manual_seed(SEED_RNG)
            v = batch_ddim_sampling(model, cond, [1, 4, T, h, w], n_samples=1, ddim_steps=STEPS, ddim_eta=1.0,
                                    cfg_scale=7.5, hs=hs, **extra)
            outs.append(v.float())
    return outs
