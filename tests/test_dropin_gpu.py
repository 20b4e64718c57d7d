"""Drop-in proof (SURVEY section 4 'integration' row, section 8b): the reference's own training and inference drivers
-- pytorch/bts_main.py and pytorch/bts_test.py, byte-for-byte unmodified -- run against OUR `bts.py`:

  1. bts_main.py trains 2 steps on a 4-image synthetic NYU-style dataset (nn.DataParallel wrap, weights_init_xavier,
     set_misc freezing by parameter name, AdamW over model.module.{encoder,decoder}, per-step loss print) and writes
     a checkpoint whose model keys carry the `module.` prefix;
  2. bts_test.py re-imports the model file by name from the checkpoint directory, loads that checkpoint into a
     DataParallel-wrapped BtsModel, runs inference and writes the 16-bit depth PNGs.

The scripts are the reference's own source, so they are never committed: `make -C oracle` copies them, unmodified, from a
checkout of the reference into the git-ignored oracle/_ref/, and the test skips where that copy is absent.
tests/dropin/boot.py supplies the environment the 2019 scripts assume (stub tensorboardX / matplotlib, two torch-2.x
compatibility shims) -- see its docstring."""
import os
import re
import shutil
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

SCRIPTS = ["bts_main.py", "bts_test.py", "bts_dataloader.py", "distributed_sampler_no_evenly_divisible.py"]


def _script_dir():
    d = os.path.join(ROOT, "oracle", "_ref")
    return d if all(os.path.isfile(os.path.join(d, s)) for s in SCRIPTS) else None


def _make_dataset(d, n=4):
    """NYU-style: <scene>/rgb_i.png (480x640 RGB) + <scene>/gt_i.png (16-bit depth, millimetres); list `rgb depth focal`
    with scene-relative paths (bts_test.py:157-164 splits them on '/')."""
    import cv2
    rng = np.random.RandomState(0)
    os.makedirs(os.path.join(d, "scene"))
    lines = []
    for i in range(n):
        yy, xx = np.mgrid[0:480, 0:640].astype(np.float32)
        img = np.stack([(xx / 640 * 255), (yy / 480 * 255), rng.uniform(0, 255, (480, 640))], -1).astype(np.uint8)
        depth_m = 1.0 + 4.0 * (yy / 480) + 0.5 * np.sin(xx / 40.0 + i)
        cv2.imwrite(os.path.join(d, "scene", "rgb_%d.png" % i), img)
        cv2.imwrite(os.path.join(d, "scene", "gt_%d.png" % i), (depth_m * 1000).astype(np.uint16))
        lines.append("scene/rgb_%d.png scene/gt_%d.png 518.8579" % (i, i))
    with open(os.path.join(d, "files.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


@pytest.mark.skipif(_script_dir() is None, reason="reference scripts not in oracle/_ref (`make -C oracle REF=<reference>/pytorch`)")
def test_unmodified_bts_main_and_bts_test_run_against_our_module(tmp_path):
    src = _script_dir()
    work = tmp_path / "work"
    work.mkdir()
    for s in SCRIPTS:
        shutil.copy(os.path.join(src, s), work / s)            # the reference's files, untouched
    shutil.copy(os.path.join(ROOT, "bts.py"), work / "bts.py")  # OUR module under the reference's module name
    data = tmp_path / "data"
    data.mkdir()
    _make_dataset(str(data))
    log = tmp_path / "log"
    log.mkdir()
    args = """--mode train
--model_name bts_dropin
--encoder densenet121_bts
--dataset nyu
--data_path {d}/
--gt_path {d}/
--filenames_file {d}/files.txt
--batch_size 2
--num_epochs 1
--learning_rate 1e-4
--weight_decay 1e-2
--adam_eps 1e-3
--num_threads 1
--input_height 128
--input_width 160
--max_depth 10
--log_directory {l}
--log_freq 1000
--save_freq 1
--data_path_eval {d}/
--gt_path_eval {d}/
--filenames_file_eval {d}/files.txt
--min_depth_eval 1e-3
--max_depth_eval 10
""".format(d=data, l=log)
    (work / "args_train.txt").write_text(args)
    env = dict(os.environ, PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), CUDA_VISIBLE_DEVICES="0",
               BTS_B200_PRETRAINED="0")
    boot = os.path.join(ROOT, "tests", "dropin", "boot.py")
    r = subprocess.run([sys.executable, boot, "bts_main.py", "args_train.txt"], cwd=work, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    losses = [float(x) for x in re.findall(r"loss: ([0-9.eE+-]+|nan|inf)", r.stdout)]
    assert len(losses) == 2 and all(np.isfinite(losses)), r.stdout[-2000:]
    assert "Fixing first conv layer" in r.stdout and "Total number of learning parameters" in r.stdout
    ckpt = log / "bts_dropin" / "model-1"
    assert ckpt.is_file(), os.listdir(log / "bts_dropin")
    assert (log / "bts_dropin" / "bts_dropin.py").is_file()       # bts_main.py copied OUR bts.py next to the checkpoint
    sd = torch.load(ckpt, map_location="cpu", weights_only=False)
    assert sd["global_step"] == 1 and all(k.startswith("module.") for k in sd["model"])
    assert "module.encoder.base_model.denseblock1.denselayer1.conv1.weight" in sd["model"]
    assert "module.decoder.reduc8x8.reduc.plane_params.weight" in sd["model"] and "optimizer" in sd

    # ---- inference driver on that checkpoint (imports bts_dropin.py from the checkpoint directory by name)
    targs = """--model_name bts_dropin
--encoder densenet121_bts
--data_path {d}/
--dataset nyu
--filenames_file {d}/files.txt
--checkpoint_path {c}
--input_height 480
--input_width 640
--max_depth 10
""".format(d=data, c=ckpt)
    (work / "args_test.txt").write_text(targs)
    r = subprocess.run([sys.executable, boot, "bts_test.py", "args_test.txt"], cwd=work, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, (r.stdout[-3000:], r.stderr[-3000:])
    assert "now testing 4 files" in r.stdout and "Done." in r.stdout
    import cv2
    raw = sorted((work / "result_bts_dropin" / "raw").glob("*.png"))
    assert len(raw) == 4
    png = cv2.imread(str(raw[0]), -1)
    assert png.dtype == np.uint16 and png.shape == (480, 640) and png.max() > 0      # depth x 1000 as uint16 (bts_test.py:179-185)
