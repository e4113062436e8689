"""Goldens for the checks that used to import the reference at test time — run with a checkout of the UNMODIFIED
reference ToonCrafter repository:

    python tests/golden/make_golden_reference_checks.py PATH/TO/ToonCrafter

Writes
  unet_seed5_reference.npz          the reference UNet's output on the tiny configuration with a second weight seed
                                    (5) and input seed (3) than make_golden.py uses (tests/test_oracle_cpu.py);
  inference_512_model_config.json   the `model` section of the reference's configs/inference_512_v1.0.yaml, as data
                                    (tests/test_oracle_cpu.py builds it with this repository's classes).
"""
import json
import sys
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(HERE.parent))

from oracle import ref_shims  # noqa: E402
from tiny_config import TINY_CONTEXT_DIM, TINY_T, TINY_UNET  # noqa: E402
from tooncrafter_b200 import modules, synthetic  # noqa: E402

WEIGHT_SEED = 5
INPUT_SEED = 3


def unet_inputs():
    """Inputs of the second-seed UNet check (shared with tests/test_oracle_cpu.py)."""
    g = torch.Generator().manual_seed(INPUT_SEED)
    x = torch.randn(1, 8, TINY_T, 16, 16, generator=g)
    ctx = torch.randn(1, 77 + 16 * TINY_T, TINY_CONTEXT_DIM, generator=g)
    return x, torch.tensor([250]), ctx, torch.tensor([7])


def main():
    ref_root = Path(sys.argv[1]).resolve()
    ref_shims.REFERENCE_ROOT = ref_root
    torch.set_num_threads(8)

    ref = ref_shims.build_reference_unet(TINY_UNET).eval()
    synthetic.fill_module_(ref, seed=WEIGHT_SEED, prefix="model.diffusion_model.")
    # the test rebuilds these weights from this repository's UNetModel: they must be the reference's, bit for bit
    mine = modules.UNetModel(**TINY_UNET)
    synthetic.fill_module_(mine, seed=WEIGHT_SEED, prefix="model.diffusion_model.")
    a, b = ref.state_dict(), mine.state_dict()
    assert set(a) == set(b) and all(torch.equal(a[k], b[k]) for k in a)
    x, t, ctx, fs = unet_inputs()
    with torch.no_grad():
        y = ref(x, t, context=ctx, fs=fs)
    np.savez_compressed(HERE / "unet_seed5_reference.npz", y=y.numpy())
    print("unet", tuple(y.shape), float(y.abs().max()))

    import yaml
    cfg = yaml.safe_load((ref_root / "configs" / "inference_512_v1.0.yaml").read_text())["model"]
    (HERE / "inference_512_model_config.json").write_text(json.dumps(cfg, indent=1) + "\n")


if __name__ == "__main__":
    main()
