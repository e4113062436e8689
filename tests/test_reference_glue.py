"""Drop-in boundary, end to end: the calls the reference's inference scripts make around the model
(scripts/evaluation/funcs.py::batch_ddim_sampling, :14-93: builds the unconditional branch, calls DDIMSampler.sample
with the kwargs the scripts really pass, both decode_first_stage passes and the middle-frame splice; restated as
tests/glue_common.py::batch_ddim_sampling) run against this repository's `lvdm.*` / `utils.*` aliases and must
reproduce what the reference's own glue produces with the unmodified reference model (tests/golden/glue_tiny.npz, made
by tests/golden/make_golden_glue.py).  Two prompts back to back (stale-conditioning regression) and one call with the
mask / x0 blending kwargs."""
import subprocess
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
STRIDE = 5


def test_batch_ddim_sampling_glue_on_the_alias_tree_matches_reference_golden(tmp_path):
    out = tmp_path / "glue_out.npz"
    r = subprocess.run([sys.executable, str(HERE / "glue_driver.py"), str(out), "cpu"], capture_output=True, text=True,
                       timeout=1500)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-4000:]
    got = np.load(out)
    gold = np.load(HERE / "golden" / "glue_tiny.npz")
    for i in range(3):
        g = gold[f"clip{i}_sub"]
        o = got[f"clip{i}"]
        assert tuple(o.shape) == tuple(gold[f"clip{i}_shape"])
        err = np.abs(o.reshape(-1)[::STRIDE] - g).max()
        scale = np.abs(g).max()
        print(f"clip {i}: max err {err:.3e} (scale {scale:.3e})")
        # fp16 activations through 4 DDIM steps + decoder on the interpreter: same bound as the other emulator tests
        assert err < 4e-2 * scale, (i, err, scale)
    # the three calls really differ (prompt 0 vs prompt 1 vs masked prompt 0)
    assert np.abs(got["clip0"] - got["clip1"]).max() > 1e-2 and np.abs(got["clip0"] - got["clip2"]).max() > 1e-2
