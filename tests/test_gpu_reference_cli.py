"""The reference's own CLIs, UNCHANGED, on the B200 engine (north star: "train.py/test.py and configs/lego.yaml
drive it unchanged"; the reference's train.py:28-102, test.py:18-55).  baseline/_ref is the unmodified checkout
staged by __graft_entry__.build() when a checkout is available (git-ignored; the test skips without it); the scripts are executed with
`python -m nerf_simple_b200.run`, which only puts the `utils` shim package in front of sys.path."""
import glob
import hashlib
import os
import re
import subprocess
import sys

import pytest
import yaml

from synth_dataset import write_dataset

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")


def _run(script, cfg, cwd):
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.path.join(ROOT, "tests"), NERF_B200_PRECISION="bf16")
    out = subprocess.run([sys.executable, "-m", "nerf_simple_b200.run", os.path.join(REF, script), "--config_path", cfg],
                         cwd=cwd, env=env, capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, (out.stdout[-3000:], out.stderr[-3000:])
    return out.stdout


@pytest.mark.skipif(not os.path.isfile(os.path.join(REF, "train.py")), reason="baseline/_ref not staged (scripts/stage_reference.sh)")
def test_reference_train_and_test_cli_unchanged(tmp_path):
    # the staged scripts are byte-identical to what stage_reference.sh hashed from the checkout
    sums = dict(reversed(ln.split()) for ln in open(os.path.join(REF, "SHA256SUMS")).read().splitlines())
    for name in ("train.py", "test.py", "utils/rendering.py", "utils/nets.py"):
        assert hashlib.sha256(open(os.path.join(REF, name), "rb").read()).hexdigest() == sums[name]
    data = write_dataset(str(tmp_path / "lego"), H=24, W=24, n_train=3, n_val=3, n_test=3)   # load_data takes num_imgs of EVERY split (utils/dataload.py:55-61)
    models, results = str(tmp_path / "models"), str(tmp_path / "results")
    cfg = yaml.safe_load(open(os.path.join(REF, "configs", "lego.yaml")))      # the reference's own config, paths/sizes shrunk
    cfg.update(datapath=data, savepath=models, exp_name="cli", num_iters=120, ckpt_model=100, ckpt_loss=10, ckpt_images=100,
               batch_size=512, Nf=32, half_res=False, val_idxs=[0], num_train_imgs=3)
    cfg_path = str(tmp_path / "cfg.yaml")
    with open(cfg_path, "w") as fh:
        yaml.safe_dump(cfg, fh)
    log = _run("train.py", cfg_path, str(tmp_path))
    losses = [float(m) for m in re.findall(r"loss: ([0-9.eE+-]+) \| epoch", log)]
    assert len(losses) == 12 and losses[-1] < 0.6 * losses[0], losses
    ckpts = sorted(glob.glob(os.path.join(models, "cli", "*.pth")))
    assert len(ckpts) >= 2                                                 # ckpt_model saves + the final save (train.py:84-91)
    assert glob.glob(os.path.join(str(tmp_path), "logs", "run_*", "events.out.tfevents.*"))   # TensorBoard scalars/images
    # test.py, still images (test.py:37-45)
    cfg["test_params"].update(batch_size=200, half_res=False, loadpath=ckpts[-1], datapath=data, savepath=results,
                              exp_name="stills", im_set="test", im_idxs=[0, 1], animation=False)
    with open(cfg_path, "w") as fh:
        yaml.safe_dump(cfg, fh)
    _run("test.py", cfg_path, str(tmp_path))
    for i in (0, 1):
        assert os.path.getsize(os.path.join(results, "stills", f"rgb_{i}.png")) > 0
        assert os.path.getsize(os.path.join(results, "stills", f"depth_{i}.png")) > 0
    # test.py, dome animation (test.py:30-35 -> render_poses -> mp4)
    cfg["test_params"].update(exp_name="anim", animation=True, num_poses=2, theta=30)
    with open(cfg_path, "w") as fh:
        yaml.safe_dump(cfg, fh)
    _run("test.py", cfg_path, str(tmp_path))
    vids = glob.glob(os.path.join(results, "anim", "nerf_rgb*.mp4"))
    assert vids and os.path.getsize(vids[0]) > 0
