"""The runner shim (cfdbench_b200/runner.py) rebinding logic, exercised on a stand-in for CFDBench's `src/` that has the
reference's module layout and seams (models/base_model.py, models/fno/fno2d.py, models/loss.py, utils/autoregressive.py,
args.py) and nothing else, written by the test so that it runs without a CFDBench checkout."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

STAND_IN = {
    # the reference ships models/ and models/fno/ without __init__.py (namespace packages), utils/ with one
    "models/base_model.py": """
        from torch import nn

        class AutoCfdModel(nn.Module):
            def __init__(self, loss_fn):
                super().__init__()
                self.loss_fn = loss_fn
        """,
    "models/loss.py": "from cfdbench_b200.loss import MseLoss, loss_name_to_fn\n",
    "models/fno/fno2d.py": """
        from ..base_model import AutoCfdModel

        class Fno2d(AutoCfdModel):
            pass
        """,
    "utils/__init__.py": "",
    "utils/autoregressive.py": "from models.fno.fno2d import Fno2d\n",
    "args.py": """
        from tap import Tap

        class Args(Tap):
            model: str = "fno"
        """,
}

CODE = r'''
import sys
sys.path.insert(0, %r)
from cfdbench_b200 import runner
runner.install(%r, stub_missing=True)
import models.fno.fno2d as ref
from models.base_model import AutoCfdModel
from models.loss import loss_name_to_fn
import cfdbench_b200.fno2d as ours
assert ref.Fno2d is ours.Fno2d, "seam not rebound"
m = ref.Fno2d(in_chan=2, out_chan=2, n_case_params=5, loss_fn=loss_name_to_fn("nmse"), num_layers=4,
              hidden_dim=32, modes1=12, modes2=12, device="cpu")
assert isinstance(m, AutoCfdModel), "must subclass the reference AutoCfdModel (test_multistep.py:109)"
assert m.loss_fn.get_score_names() == ["mse", "rmse", "mae", "nmse"]
# the factory the scripts use picks the rebound class up (utils/autoregressive.py:10,114-125)
import utils.autoregressive as ua
assert ua.Fno2d is ours.Fno2d
import args
assert args.Args.lr_step_size == 20, "train_auto.py reads args.lr_step_size, which Args does not declare"
print("ok")
'''


def test_runner_rebinds_the_seam_and_subclasses_reference_base(tmp_path):
    src = tmp_path / "src"
    for rel, body in STAND_IN.items():
        (src / rel).parent.mkdir(parents=True, exist_ok=True)
        (src / rel).write_text(textwrap.dedent(body).lstrip())
    out = subprocess.run([sys.executable, "-c", CODE % (ROOT, str(src))], capture_output=True, text=True,
                         env={**os.environ, "PYTHONDONTWRITEBYTECODE": "1"})
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip().endswith("ok"), out.stdout
