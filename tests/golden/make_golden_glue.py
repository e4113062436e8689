"""Golden for the reference-glue integration test: the UNMODIFIED reference's scripts/evaluation/funcs.py::
batch_ddim_sampling driving the UNMODIFIED reference model (tiny configuration, CPU fp32) — run with a checkout of the
reference ToonCrafter repository:

    python tests/golden/make_golden_glue.py PATH/TO/ToonCrafter
"""
import importlib.util
import sys
import types
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(HERE.parent))

from oracle import ref_shims  # noqa: E402
from tiny_config import TINY_CONTEXT_DIM, TINY_LATENT_HW, TINY_T, model_config  # noqa: E402
from tooncrafter_b200 import synthetic  # noqa: E402
import glue_common  # noqa: E402

STRIDE = 5


def load_reference_funcs(ref_root):
    """The reference's scripts/evaluation/funcs.py, loaded by file; decord / cv2 are video-I/O imports at its top
    (absent here, never called on this path)."""
    for name in ("decord", "cv2"):
        if name not in sys.modules:
            m = types.ModuleType(name)
            m.VideoReader = m.cpu = None
            sys.modules[name] = m
    spec = importlib.util.spec_from_file_location("reference_eval_funcs", ref_root / "scripts" / "evaluation" / "funcs.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def main():
    ref_root = Path(sys.argv[1]).resolve()
    ref_shims.REFERENCE_ROOT = ref_root
    torch.set_num_threads(8)
    model = ref_shims.build_reference_model(model_config()).eval()
    synthetic.fill_module_(model, seed=0)
    model.perframe_ae = True
    model.temporal_length = TINY_T
    # harness shim 3 (SURVEY 8c): the reference sampler hard-codes "cuda" in register_buffer (ddim.py:18-22)
    import lvdm.models.samplers.ddim as ref_ddim

    def register_buffer(self, name, attr):
        if isinstance(attr, torch.Tensor):
            attr = attr.to(self.model.device)
        setattr(self, name, attr)
    ref_ddim.DDIMSampler.register_buffer = register_buffer
    funcs = load_reference_funcs(ref_root)
    assert funcs.DDIMSampler is ref_ddim.DDIMSampler
    outs = glue_common.run_glue(funcs.batch_ddim_sampling, model, TINY_T, *TINY_LATENT_HW, TINY_CONTEXT_DIM)
    save = {}
    for i, o in enumerate(outs):
        save[f"clip{i}_sub"] = o.flatten()[::STRIDE].numpy()
        save[f"clip{i}_shape"] = np.array(o.shape)
        print(i, tuple(o.shape), float(o.abs().max()))
    np.savez_compressed(HERE / "glue_tiny.npz", **save)


if __name__ == "__main__":
    main()
