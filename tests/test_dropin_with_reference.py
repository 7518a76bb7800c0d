"""CPU: the sys.path shadowing of INTEGRATION.md §1 resolves `models.pose_mobilenet` / `core.group` /
`utils.transforms` to this repo and `core.inference`, `utils.zipreader` ... to the reference, and the reference glue
runs on our module's outputs.  The reference is a stand-in tree with the reference's package layout (written per test):
`lib/models` a regular package that imports its members, `lib/core` and `lib/utils` namespace packages, `_init_paths.py`
putting `lib` at the front of sys.path; its `core.inference` is the glue restatement oracle/glue_ref.py."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STAND_IN = {
    "_init_paths.py": "import os.path, sys\n"
                      "lib = os.path.join(os.path.dirname(__file__), 'lib')\n"
                      "if lib not in sys.path:\n    sys.path.insert(0, lib)\n",
    "lib/models/__init__.py": "import models.pose_higher_hrnet\nimport models.pose_mobilenet\n",
    "lib/models/pose_higher_hrnet.py": "def get_pose_net(cfg, is_train, **kwargs):\n    raise NotImplementedError\n",
    "lib/models/pose_mobilenet.py": "raise ImportError('the stand-in reference model must never be imported')\n",
    "lib/core/group.py": "raise ImportError('the stand-in reference parser must never be imported')\n",
    "lib/core/inference.py": "from dataset.transforms import FLIP_CONFIG\n"
                             "from oracle.glue_ref import aggregate_results\n"
                             "from oracle.glue_ref import multi_stage_outputs as get_multi_stage_outputs\n",
    "lib/utils/transforms.py": "def fliplr_joints(joints, joints_vis, width, matched_parts):\n"
                               "    raise NotImplementedError\n",
    "lib/utils/zipreader.py": "def imread(filename):\n    raise NotImplementedError\n",
}


@pytest.fixture
def ref_tree(tmp_path):
    base = tmp_path / "reference"
    for rel, text in STAND_IN.items():
        path = base / rel
        path.parent.mkdir(parents=True, exist_ok=True)
        path.write_text(text)
    return str(base)

SCRIPT = r'''
import sys, types
sys.path.insert(0, "%(ref)s/lib"); sys.path.insert(0, "%(ref)s")
sys.path.insert(0, "%(root)s"); sys.path.insert(0, "%(root)s/litepose_b200/lib")
from litepose_b200.config import FLIP_CONFIG, get_cfg, get_arch
ds = types.ModuleType("dataset"); dst = types.ModuleType("dataset.transforms"); dst.FLIP_CONFIG = FLIP_CONFIG
ds.transforms = dst; sys.modules["dataset"] = ds; sys.modules["dataset.transforms"] = dst
import torch, models
from core.group import HeatmapParser
from core.inference import get_multi_stage_outputs, aggregate_results
assert "litepose_b200" in models.pose_mobilenet.__file__, models.pose_mobilenet.__file__
assert "litepose_b200" in sys.modules["core.group"].__file__
assert "%(ref)s" in sys.modules["core.inference"].__file__
cfg = get_cfg(input_size=64)
model = eval("models." + cfg.MODEL.NAME + ".get_pose_net")(cfg, is_train=True, cfg_arch=get_arch("XS")).eval()
with torch.no_grad():
    o, h, t = get_multi_stage_outputs(cfg, model, torch.rand(1, 3, 64, 64), True, True, (64, 64))
    fh, tl = aggregate_results(cfg, 1, None, [], h, t)
assert tuple(fh.shape) == (1, 14, 64, 64) and tuple(torch.cat(tl, 4).shape) == (1, 14, 64, 64, 2)
HeatmapParser(cfg)
# valid.py:44-46 and :27-29: the coordinate helpers come from this repo, the other utils modules from the reference
from utils.transforms import resize_align_multi_scale, get_final_preds, get_multi_scale_size
import utils.transforms, utils.zipreader
assert "litepose_b200" in utils.transforms.__file__ and "%(ref)s" in utils.zipreader.__file__
assert utils.transforms.fliplr_joints.__module__ == "_reference_utils_transforms"      # delegated, not restated
import numpy as np
size, center, scale = get_multi_scale_size(np.zeros((480, 640, 3), np.uint8), 512, 1.0, 1.0)
assert size == (704, 512) and list(center) == [320, 240]
print("dropin ok")
'''


def test_sys_path_shadowing(ref_tree):
    r = subprocess.run([sys.executable, "-c", SCRIPT % {"ref": ref_tree, "root": ROOT}], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0 and "dropin ok" in r.stdout, r.stdout + r.stderr


CHECK = r'''
import sys, types
import _init_paths                                   # what valid.py:24 does: <reference>/lib to the FRONT of sys.path
assert sys.path[0].endswith("lib"), sys.path[:3]
from litepose_b200.config import FLIP_CONFIG
ds = types.ModuleType("dataset"); dst = types.ModuleType("dataset.transforms"); dst.FLIP_CONFIG = FLIP_CONFIG
ds.transforms = dst; sys.modules["dataset"] = ds; sys.modules["dataset.transforms"] = dst
import models
from core.group import HeatmapParser
from core.inference import get_multi_stage_outputs
from utils.transforms import get_final_preds
import utils.zipreader
repo = "%(root)s"
assert models.pose_mobilenet.__file__.startswith(repo), models.pose_mobilenet.__file__
assert sys.modules["core.group"].__file__.startswith(repo)
assert sys.modules["utils.transforms"].__file__.startswith(repo)
assert sys.modules["core.inference"].__file__.startswith("%(ref)s")
assert utils.zipreader.__file__.startswith("%(ref)s")
import models.pose_higher_hrnet as hr                # the rest of the model zoo still comes from the reference
assert hr.__file__.startswith("%(ref)s")
print("init_paths dropin ok")
'''


@pytest.mark.parametrize("how", ["sitecustomize", "runner"])
def test_dropin_survives_init_paths(tmp_path, ref_tree, how):
    """ADVICE r1: valid.py's `import _init_paths` inserts <reference>/lib at sys.path[0] AFTER PYTHONPATH /
    sitecustomize, and <reference>/lib/models is a regular package - plain path shadowing loses and the model would
    silently be the stock eager one.  The meta-path drop-in (litepose_b200/dropin.py) must win in both launch modes."""
    script = tmp_path / "check_like_valid.py"
    script.write_text(CHECK % {"ref": ref_tree, "root": ROOT})
    env = dict(os.environ)
    if how == "sitecustomize":
        env["PYTHONPATH"] = os.pathsep.join([os.path.join(ROOT, "litepose_b200", "dropin_site"), ROOT])
        # cwd = reference root so that `import _init_paths` resolves like for `python valid.py`
        cmd = [sys.executable, "-c", "import sys; sys.path.insert(0, %r); exec(open(%r).read())" % (ref_tree, str(script))]
    else:
        env["PYTHONPATH"] = ROOT
        # the runner puts the script's directory first (as `python script.py` does); _init_paths lives beside valid.py
        link = tmp_path / "ref"
        os.symlink(ref_tree, link)
        runner_script = tmp_path / "run_in_ref.py"
        runner_script.write_text("import sys; sys.path.insert(0, %r)\n" % ref_tree + CHECK % {"ref": ref_tree, "root": ROOT})
        cmd = [sys.executable, "-m", "litepose_b200.dropin", str(runner_script)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=env, cwd=ref_tree)
    assert r.returncode == 0 and "init_paths dropin ok" in r.stdout, r.stdout + r.stderr
