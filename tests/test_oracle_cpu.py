"""CPU tests (no GPU): the oracle (oracle/*.py, our restatement of the reference algorithm) against the committed
golden outputs of the UNMODIFIED reference (tests/golden/, made by make_golden.py and
make_golden_reference_checks.py), plus host-side logic: schedule known answers, state-dict key compatibility, the
reference's inference config, C-ABI symbol export.
"""
import json
import sys
from pathlib import Path

import numpy as np
import pytest
import torch

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE))
sys.path.insert(0, str(HERE / "golden"))

from tiny_config import (FULL_DDCONFIG, FULL_UNET, TINY_CONTEXT_DIM, TINY_DDCONFIG, TINY_LATENT_HW, TINY_T,  # noqa: E402
                         TINY_UNET)
from make_golden import SEED, golden_inputs  # noqa: E402

from oracle import ddim_oracle, unet_oracle, vae_oracle  # noqa: E402
from tooncrafter_b200 import layout, modules, synthetic  # noqa: E402

GOLD = np.load(HERE / "golden" / "tiny_reference_outputs.npz")
KAT = json.loads((HERE / "golden" / "schedule_kat.json").read_text())


@pytest.fixture(scope="module")
def tiny_sd():
    """Seeded synthetic weights under the reference checkpoint's key names (tiny config)."""
    man = json.loads((HERE / "golden" / "state_dict_manifest_tiny.json").read_text())
    sched = ddim_oracle.model_schedule()
    sd = {}
    for k, shape in man.items():
        if k.startswith(("model.", "first_stage_model.")):
            sd[k] = synthetic.synthetic_tensor(k, tuple(shape), SEED)
    sd.update({k: v for k, v in sched.items()})
    return sd


def _close(a, b, tol):
    a = torch.as_tensor(a).float()
    b = torch.as_tensor(b).float()
    assert a.shape == b.shape
    err = (a - b).abs().max().item()
    assert err <= tol * max(1.0, b.abs().max().item()), f"max err {err:.3e}"


def test_schedule_known_answers():
    sched = ddim_oracle.model_schedule()
    assert KAT["scale_arr_len"] == 1400 and sched["scale_arr"].shape[0] == 1400
    assert list(ddim_oracle.ddim_timesteps(50)) == KAT["ddim_timesteps_50"]
    assert list(ddim_oracle.ddim_timesteps(10)) == KAT["ddim_timesteps_10"]
    assert KAT["ddim_timesteps_50"][:3] == [19, 39, 59] and KAT["ddim_timesteps_50"][-1] == 999
    assert KAT["ddim_timesteps_10"] == [99 + 100 * i for i in range(10)]
    tab = ddim_oracle.ddim_tables(sched, 50, 1.0)
    assert abs(float(tab["alphas_prev"][-1]) - KAT["a_prev_last"]) < 1e-12
    assert abs(float(tab["sigmas"][-1]) - KAT["sigma_last"]) < 1e-12
    assert float(sched["alphas_cumprod"][-1]) == 0.0 == KAT["alphas_cumprod_last"]
    assert abs(float(sched["alphas_cumprod"][0]) - 0.99915) < 1e-5
    assert abs(float(sched["scale_arr"][999]) - 0.7) < 1e-7 and abs(float(sched["scale_arr"][19]) - 0.985714) < 1e-6
    for k in ("betas", "alphas_cumprod", "sqrt_alphas_cumprod", "sqrt_one_minus_alphas_cumprod", "scale_arr"):
        assert np.array_equal(sched[k].numpy(), GOLD["sched_" + k]), k
    # first step: direction coefficient sqrt(1 - a_prev - sigma^2) in fp32 (SURVEY App. C.11)
    co = ddim_oracle.step_coefficients(sched, tab, 49)
    assert co["sqrt_ac"] == 0.0 and co["sqrt_1mac"] == 1.0
    assert abs(co["dir_coef"] - 5.96e-8 ** 0.5) < 1e-6
    co10 = ddim_oracle.step_coefficients(sched, ddim_oracle.ddim_tables(sched, 10, 1.0), 9)
    assert co10["dir_coef"] == 0.0


def test_unet_oracle_matches_reference_golden(tiny_sd):
    gi = golden_inputs()["unet"]
    y = unet_oracle.unet_forward(tiny_sd, layout.unet_layout(TINY_UNET), gi["x"], gi["t"], gi["ctx"], gi["fs"],
                                 prefix="model.diffusion_model.")
    _close(y, GOLD["unet_y"], 2e-5)


def test_vae_oracle_matches_reference_golden(tiny_sd):
    gi = golden_inputs()
    moments, hidden = vae_oracle.encode_hidden(tiny_sd, layout.encoder_layout(TINY_DDCONFIG), gi["frames"])
    for i, h in enumerate(hidden):
        _close(h.flatten()[::97], GOLD[f"enc_hidden{i}_sub"], 2e-5)
    ref_ctx = [h.reshape(1, 2, *h.shape[1:]).permute(0, 2, 1, 3, 4) for h in hidden]
    dec = vae_oracle.decode_first_stage(tiny_sd, layout.decoder_layout(TINY_DDCONFIG), gi["z"], ref_ctx, chunk=TINY_T)
    _close(dec, GOLD["decode"], 2e-5)


def test_ddim_oracle_matches_reference_golden(tiny_sd):
    gi = golden_inputs()
    ulay = layout.unet_layout(TINY_UNET)

    def apply_model(x, t, c, fs):
        xc = torch.cat([x] + c["c_concat"], dim=1)
        cc = torch.cat(c["c_crossattn"], dim=1)
        return unet_oracle.unet_forward(tiny_sd, ulay, xc, t, cc, fs, prefix="model.diffusion_model.")

    x, _ = ddim_oracle.sample(apply_model, ddim_oracle.model_schedule(), gi["x_T"], gi["cond"], gi["uncond"], gi["S"],
                              noises=gi["noises"], fs=gi["fs"])
    _close(x, GOLD["ddim_samples"], 2e-4)


def test_state_dict_keys_match_reference_manifest():
    """Our parameter holders expose exactly the reference checkpoint's keys/shapes (full 512 model)."""
    man = json.loads((HERE / "golden" / "state_dict_manifest_512.json").read_text())
    with torch.device("meta"):
        unet = modules.UNetModel(**FULL_UNET)
        dec = modules.VideoDecoder(**FULL_DDCONFIG)
        enc = modules.Encoder(**FULL_DDCONFIG)
    mine = {"model.diffusion_model." + k: list(v.shape) for k, v in unet.state_dict().items()}
    mine.update({"first_stage_model.decoder." + k: list(v.shape) for k, v in dec.state_dict().items()})
    mine.update({"first_stage_model.encoder." + k: list(v.shape) for k, v in enc.state_dict().items()})
    ref = {k: v for k, v in man.items() if k.startswith(tuple(p for p in ("model.diffusion_model.",
                                                                          "first_stage_model.decoder.",
                                                                          "first_stage_model.encoder.")))}
    assert set(mine) == set(ref)
    bad = [k for k in ref if mine[k] != ref[k]]
    assert not bad, bad[:5]
    assert len([k for k in ref if k.startswith("model.diffusion_model.")]) == 1516
    assert "model.diffusion_model.input_blocks.1.0.temopral_conv.conv1.2.weight" in mine   # load-bearing typo


def test_c_abi_library_exports_every_declared_symbol():
    """The .so loads on a GPU-less host and exports every symbol include/tooncrafter_b200.h declares."""
    import re
    from tooncrafter_b200 import _lib
    header = (HERE.parent / "include" / "tooncrafter_b200.h").read_text()
    declared = set(re.findall(r"\b(tc_[a-z0-9_]+)\s*\(", header))
    lib = _lib.load()
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in the header but not exported"
    assert declared == set(_lib.EXPORTED_SYMBOLS)
    assert lib.tc_version() >= 100


def test_unet_oracle_matches_reference_golden_second_seed():
    """The oracle against the unmodified reference UNet with other weight / input seeds than the goldens above
    (tests/golden/unet_seed5_reference.npz, made by make_golden_reference_checks.py)."""
    from make_golden_reference_checks import WEIGHT_SEED, unet_inputs
    unet = modules.UNetModel(**TINY_UNET)
    synthetic.fill_module_(unet, seed=WEIGHT_SEED, prefix="model.diffusion_model.")
    sd = {"model.diffusion_model." + k: v for k, v in unet.state_dict().items()}
    x, t, ctx, fs = unet_inputs()
    with torch.no_grad():
        b = unet_oracle.unet_forward(sd, layout.unet_layout(TINY_UNET), x, t, ctx, fs, "model.diffusion_model.")
    a = torch.from_numpy(np.load(HERE / "golden" / "unet_seed5_reference.npz")["y"])
    assert a.shape == b.shape
    err = (a - b).abs().max().item()
    assert err < 2e-5, err


def test_reference_yaml_config_builds_our_classes_with_checkpoint_keys():
    """The `model` section of the reference's own configs/inference_512_v1.0.yaml (stored as
    tests/golden/inference_512_model_config.json), fed to OUR instantiate_from_config with this repository first on the
    import path (INTEGRATION.md 1): every hot-path `target:` resolves to our classes, their constructors accept the
    YAML's kwargs, and the resulting state dict carries the public checkpoint's keys.  Only the two OpenCLIP towers (out
    of scope, need network weights) are swapped for Identity."""
    cfg = json.loads((HERE / "golden" / "inference_512_model_config.json").read_text())
    for k in ("cond_stage_config", "img_cond_stage_config"):
        cfg["params"][k] = {"target": "torch.nn.Identity"}
    cfg["params"]["unet_config"]["params"]["use_checkpoint"] = False            # inference.py:286
    from tooncrafter_b200 import diffusion
    with torch.device("meta"):
        m = diffusion.instantiate_from_config(cfg)
    assert type(m).__module__ == "tooncrafter_b200.diffusion" and type(m).__name__ == "LatentVisualDiffusion"
    assert type(m.model.diffusion_model).__module__ == "tooncrafter_b200.modules"
    assert type(m.first_stage_model).__name__ == "AutoencoderKL_Dualref"
    assert type(m.image_proj_model).__module__ == "tooncrafter_b200.modules"      # lvdm.modules.encoders.resampler alias
    assert m.perframe_ae and m.model.conditioning_key == "hybrid" and m.temporal_length == 16
    sd = {k: list(v.shape) for k, v in m.state_dict().items()}
    man = json.loads((HERE / "golden" / "state_dict_manifest_512.json").read_text())
    missing = [k for k in man if k not in sd]
    assert not missing, missing[:5]                                               # every UNet / VAE / schedule key
    assert all(sd[k] == man[k] for k in man)
    rs = json.loads((HERE / "golden" / "state_dict_manifest_resampler.json").read_text())
    assert {k: sd["image_proj_model." + k] for k in rs} == rs


def test_missing_cuda_library_fails_loudly(monkeypatch, tmp_path):
    """No CPU fallback: without the built .so (and without a way to build it) loading raises, it does not degrade."""
    from tooncrafter_b200 import _lib, build as _build
    monkeypatch.setattr(_lib, "_LIB", None)
    monkeypatch.setattr(_lib, "lib_path", lambda: tmp_path / "libtooncrafter_b200.so")
    monkeypatch.setattr(_build, "build", lambda *a, **k: (_ for _ in ()).throw(RuntimeError("nvcc not found")))
    with pytest.raises(_lib.TcError):
        _lib.load()
    # and the engines refuse to run anywhere but on a GPU
    from tooncrafter_b200.engine import UNetEngine
    from tiny_config import TINY_UNET
    with pytest.raises(RuntimeError):
        UNetEngine(modules.UNetModel(**TINY_UNET))


def test_product_code_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under tooncrafter_b200/, lvdm/ or utils/ may import it."""
    import re
    root = HERE.parent
    offenders = []
    for d in ("tooncrafter_b200", "lvdm", "utils"):
        for f in (root / d).rglob("*.py"):
            src = f.read_text()
            if re.search(r"^\s*(from|import)\s+oracle\b", src, re.M) or "import_module(\"oracle" in src:
                offenders.append(str(f.relative_to(root)))
    assert not offenders, offenders


def test_utils_alias_covers_the_reference_surface():
    """utils/utils.py shadows the reference's module when this repo is ahead on PYTHONPATH, so it must export every
    public function of the reference file (lvdm/modules/encoders/condition.py imports count_params from it)."""
    import importlib
    # every top-level function of the reference's utils/utils.py
    names = {"count_params", "check_istarget", "instantiate_from_config", "get_obj_from_str", "load_npz_from_dir",
             "load_npz_from_paths", "resize_numpy_image", "setup_dist"}
    sys.modules.pop("utils.utils", None)
    sys.modules.pop("utils", None)
    mod = importlib.import_module("utils.utils")
    assert Path(mod.__file__).resolve().parent.parent == Path(__file__).resolve().parent.parent
    missing = sorted(n for n in names if not hasattr(mod, n))
    assert not missing, f"utils.utils alias lacks {missing}"
    assert mod.count_params(torch.nn.Linear(3, 4)) == 16
    assert mod.check_istarget("a.b.attn2.to_k", ["attn2"]) and not mod.check_istarget("a.b", ["zz"])
