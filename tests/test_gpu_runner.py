"""The reference's own scripts, UNCHANGED, on the drop-in (north_star: "train_auto.py and test_multistep.py run unchanged").

The scripts come from `oracle/_ref/src`, the unmodified reference tree byte-compiled there by `__graft_entry__.build()`
(oracle/build_ref.py), or from a CFDBench `src/` directory named by CFDBENCH_SRC; the tests skip when neither exists.
`python -m cfdbench_b200.runner <src> <script> --stub-missing ...` rebinds the plug-in seam
(reference src/utils/autoregressive.py:10) and runs the script as `__main__`; stand-ins are installed only for packages
this image lacks (tap, matplotlib, diffusers, ...).  Data: a tiny on-disk cavity set in the reference's format
(tools/make_tiny_cavity.py; reference src/dataset/cavity.py:15-34).

Covers reference src/train_auto.py:181-313 (train loop, evaluate() under torch.inference_mode() :86, preds.view :106,
StepLR :214-216,280, checkpoint save :301), :126-152 (test) and src/test_multistep.py:102-236 (generate_many rollouts,
per-step metrics, load_best_ckpt)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = os.path.abspath(os.environ.get("CFDBENCH_SRC") or os.path.join(ROOT, "oracle", "_ref", "src"))

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not os.path.isdir(os.path.join(REF_SRC, "models", "fno")),
                                 reason="no reference tree: oracle/_ref/src was not built and CFDBENCH_SRC is unset")]

COMMON = ["--model", "fno", "--data_name", "cavity_prop_bc_geo", "--loss_name", "nmse", "--lr", "0.001"]


def run_script(script, data_dir, out_dir, extra, act=None):
    if not os.path.exists(os.path.join(REF_SRC, script)):
        script += "c"   # the byte-compiled tree holds train_auto.pyc, ...
    cmd = [sys.executable, "-m", "cfdbench_b200.runner", REF_SRC, script, "--stub-missing"]
    if act:
        cmd += ["--act-dtype", act]
    cmd += COMMON + ["--data_dir", data_dir, "--output_dir", out_dir] + extra
    env = {**os.environ, "PYTHONPATH": ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""), "PYTHONDONTWRITEBYTECODE": "1"}
    return subprocess.run(cmd, capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)


@pytest.fixture(scope="module")
def tiny(tmp_path_factory):
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_tiny_cavity
    d = tmp_path_factory.mktemp("tinydata")
    make_tiny_cavity.make(str(d))
    return str(d)


@pytest.mark.parametrize("act", [None, "bfloat16"])
def test_train_auto_and_test_multistep_run_unchanged(tiny, tmp_path, act):
    out = str(tmp_path / "result")
    r = run_script("train_auto.py", tiny, out, ["--num_epochs", "2", "--batch_size", "4", "--eval_batch_size", "2",
                                                "--eval_interval", "1", "--log_interval", "2", "--mode", "train_test"], act)
    assert r.returncode == 0, (r.stdout[-1500:], r.stderr[-3000:])
    assert "====== Training done ======" in r.stdout and "=== Testing done ===" in r.stdout
    run_dir = os.path.join(out, "auto", "cavity_prop_bc_geo", "dt0.1", "fno", "lr0.001_d4_h32_m112_m212")
    assert os.path.isdir(run_dir), os.listdir(out)
    losses = json.load(open(os.path.join(run_dir, "train_losses.json")))
    assert len(losses) >= 4 and all(np.isfinite(losses))
    assert np.mean(losses[len(losses) // 2:]) < np.mean(losses[:len(losses) // 2])   # Adam at lr 1e-3 makes progress
    for ep in (0, 1):
        ck = os.path.join(run_dir, f"ckpt-{ep}")
        sc = json.load(open(os.path.join(ck, "scores.json")))
        assert np.isfinite(sc["dev_loss"]) and np.isfinite(sc["train_loss"])
        dev = json.load(open(os.path.join(ck, "dev_scores.json")))
        assert set(dev["mean"]) >= {"mse", "nmse", "mae", "rmse", "input_nmse"}
    test_scores = json.load(open(os.path.join(run_dir, "test", "scores.json")))
    assert np.isfinite(test_scores["mean"]["nmse"])
    preds = torch.load(os.path.join(run_dir, "test", "preds.pt"))
    assert preds.dim() == 4 and tuple(preds.shape[1:]) == (1, 64, 64)   # evaluate(): preds.view(-1, 1, h, w)

    # the checkpoint the drop-in wrote is the reference's checkpoint ABI: load it into the UNMODIFIED reference module and
    # compare its CPU forward with the drop-in's GPU forward on the same frame
    ckpt = os.path.join(run_dir, "ckpt-1", "model.pt")
    code = f"""
import sys, json, torch, numpy as np
sys.path.insert(0, {REF_SRC!r}); sys.path.insert(0, {ROOT!r})
from models.fno.fno2d import Fno2d as Ref
from models.loss import loss_name_to_fn
sd = torch.load({ckpt!r}, map_location="cpu")
ref = Ref(in_chan=2, out_chan=2, n_case_params=5, loss_fn=loss_name_to_fn("nmse"), num_layers=4, hidden_dim=32, modes1=12, modes2=12)
ref.load_state_dict(sd); ref.eval()
from cfdbench_b200 import Fno2d, loss_name_to_fn as ours_loss
m = Fno2d(in_chan=2, out_chan=2, n_case_params=5, loss_fn=ours_loss("nmse"), num_layers=4, hidden_dim=32, modes1=12, modes2=12)
m.load_state_dict(sd)
g = torch.Generator().manual_seed(0)
x = torch.randn(2, 2, 64, 64, generator=g); cp = torch.randn(2, 5, generator=g); mk = torch.ones(2, 1, 64, 64)
with torch.no_grad():
    a = ref.generate(inputs=x, case_params=cp, mask=mk)
    b = m.generate(x.cuda(), cp.cuda(), mk.cuda()).cpu()
print(json.dumps(dict(rel=float((a - b).norm() / a.norm()))))
"""
    r2 = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r2.returncode == 0, r2.stderr[-2000:]
    assert json.loads(r2.stdout.strip().splitlines()[-1])["rel"] < 1e-5

    r3 = run_script("test_multistep.py", tiny, out, [], act)
    assert r3.returncode == 0, (r3.stdout[-1500:], r3.stderr[-3000:])
    metrics = json.load(open(os.path.join(run_dir, "multistep_metrics.json")))
    assert len(metrics) == 20 and all(np.isfinite(m_["nmse"]) and np.isfinite(m_["mse"]) for m_ in metrics)
