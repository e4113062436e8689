"""Runs glue_common.batch_ddim_sampling — the calls the reference's inference scripts make around the model — against
this repository's alias tree (`lvdm.*` -> tooncrafter_b200) on the tiny configuration and saves the decoded clips.
Executed in a fresh interpreter by tests/test_reference_glue.py with this repository first on sys.path (so the glue's
`from lvdm.models.samplers.ddim import DDIMSampler` and the YAML targets resolve to the aliases).

    python tests/glue_driver.py OUT.npz [cpu|cuda]

On a CPU-only host the engines' recorded programs are interpreted by tests/ops_emulator.py (host-logic check); with a
GPU the CUDA kernels run."""
import sys
from pathlib import Path

import numpy as np
import torch

HERE = Path(__file__).resolve().parent
ROOT = HERE.parent
sys.path[:0] = [str(ROOT), str(HERE)]


def main():
    out, dev = sys.argv[1], (sys.argv[2] if len(sys.argv) > 2 else "cpu")
    import glue_common
    from tiny_config import TINY_CONTEXT_DIM, TINY_LATENT_HW, TINY_T, model_config
    from tooncrafter_b200 import runtime, synthetic
    from utils.utils import instantiate_from_config            # the alias (plugin seam)
    import lvdm.models.samplers.ddim as alias_ddim
    assert Path(alias_ddim.__file__).resolve().is_relative_to(ROOT), "lvdm.* must resolve to this repository's aliases"
    if dev == "cpu":
        import ops_emulator
        runtime.TEST_EXECUTOR = ops_emulator.executor
        # the interpreted programs are many small host ops: they stop scaling long before the core count of a large
        # host, where oversubscribed threads make them slower instead
        torch.set_num_threads(min(torch.get_num_threads(), 16))
    model = instantiate_from_config(model_config()).eval()
    synthetic.fill_module_(model, seed=0)
    model.perframe_ae = True
    model.temporal_length = TINY_T
    model = model.to(dev)

    # glue_common builds CPU inputs / doubles: move what the glue hands to the model onto the model's device
    real_run = glue_common.glue_inputs

    def inputs_on_device(*a):
        gi = real_run(*a)
        mv = lambda v: v.to(dev) if isinstance(v, torch.Tensor) else ([t.to(dev) for t in v] if isinstance(v, list) else v)
        return {k: mv(v) for k, v in gi.items()}
    glue_common.glue_inputs = inputs_on_device
    real_doubles = glue_common.install_conditioning_doubles

    def doubles_on_device(m, T, C):
        real_doubles(m, T, C)
        glc, emb, proj = m.get_learned_conditioning, m.embedder, m.image_proj_model
        m.get_learned_conditioning = lambda p: glc(p).to(dev)
        m.embedder = glue_common._Fn(lambda img: emb(img).to(dev))
        m.image_proj_model = glue_common._Fn(lambda t: proj(t.cpu()).to(dev))
    glue_common.install_conditioning_doubles = doubles_on_device
    outs = glue_common.run_glue(glue_common.batch_ddim_sampling, model, TINY_T, *TINY_LATENT_HW, TINY_CONTEXT_DIM)
    np.savez_compressed(out, **{f"clip{i}": o.float().cpu().numpy() for i, o in enumerate(outs)})
    print("glue ok", [tuple(o.shape) for o in outs])


if __name__ == "__main__":
    main()
