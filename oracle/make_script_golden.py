"""Generate tests/golden/inference_script_run.json and tests/golden/inference_script_image.npz by executing the reference's
unmodified `inference_IMAGdressing.py` as `__main__` against this repo's drop-ins (tests/test_reference_script_cpu.py
describes the set-up and replays the recorded call):

    python oracle/make_script_golden.py <reference source tree>

The script runs on the CPU with the kernel wrappers emulated in torch (tests/emulated_ops.py), in a temporary working
directory that holds the small random-init hub models and checkpoint the test builds.
"""
import json
import os
import runpy
import sys
import tempfile

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import emulated_ops  # noqa: E402
import test_reference_script_cpu as t  # noqa: E402


def main(reference):
    script = os.path.join(os.path.abspath(reference), "inference_IMAGdressing.py")
    import imagdressing_b200.pipelines as pl

    with tempfile.TemporaryDirectory() as tmp, pytest.MonkeyPatch.context() as mp:
        emulated_ops.install(mp)
        unet = t.make_hub(tmp)
        ckpt = t.make_checkpoint(tmp, unet)
        cloth = t.make_cloth(os.path.join(tmp, "cloth.png"))
        # the stand-in diffusers is opt-in: visible only while the script runs
        mp.syspath_prepend(os.path.join(ROOT, "imagdressing_b200", "compat"))
        mp.syspath_prepend(ROOT)
        for m in [m for m in sys.modules if m == "diffusers" or m.startswith("diffusers.")]:
            mp.delitem(sys.modules, m)
        mp.chdir(tmp)
        mp.setenv("HF_HUB_OFFLINE", "1")
        mp.setattr(sys, "argv", ["inference_IMAGdressing.py", "--cloth_path", cloth, "--model_ckpt", ckpt,
                                 "--output_path", os.path.join(tmp, "out"), "--device", "cpu"])
        seen = {}
        real_run = pl._DressingPipelineBase._run

        def spy(self, **kw):
            seen["run"] = t.describe_run(self, kw)
            out = real_run(self, **kw)
            seen["image"] = np.asarray(out.images[0])
            return out

        mp.setattr(pl._DressingPipelineBase, "_run", spy)
        try:
            runpy.run_path(script, run_name="__main__")
        finally:
            for m in [m for m in sys.modules if m == "diffusers" or m.startswith("diffusers.")]:
                sys.modules.pop(m, None)
        from PIL import Image

        grid = np.asarray(Image.open(os.path.join(tmp, "out", "cloth.png")))
        # the saved grid is [garment | generated image]
        assert grid.shape == (640, 1024, 3) and np.array_equal(grid[:, 512:], seen["image"]), grid.shape
    gold = os.path.join(ROOT, "tests", "golden")
    with open(os.path.join(gold, "inference_script_run.json"), "w") as f:
        json.dump(seen["run"], f, indent=1, sort_keys=True)
        f.write("\n")
    np.savez_compressed(os.path.join(gold, "inference_script_image.npz"), **t.image_summary(seen["image"]))


if __name__ == "__main__":
    main(sys.argv[1])
