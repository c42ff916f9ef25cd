"""Drop-in check: the REFERENCE's own, unmodified `train.py` runs against this framework - its `import internlm...` lines resolve to
`internevo_b200` through the alias package - and trains the demo config on 2 CPU ranks to the same losses as our `train.py`.  The
losses of the reference's script are stored under `tests/golden/reference` (nothing of the script lives in this repo);
`INTERNEVO_REFERENCE=<checkout of the reference>` runs it again (from pytest's temp dir, so that the script's directory does not
put the reference package first on `sys.path`) and rewrites them."""
import json
import os
import re
import subprocess
import sys


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _losses(script, port, cwd):
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", PYTHONPATH=ROOT + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", str(port), script, "--config", os.path.join(ROOT, "configs", "demo.py"),
                        "--launcher", "torch", "--backend", "gloo"], cwd=cwd, capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, (r.stdout + r.stderr)[-3000:]
    return [float(x) for x in re.findall(r"step=\d+ loss=([0-9.]+)", r.stdout + r.stderr)]


def test_reference_train_py_runs_on_this_framework(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from common import find_free_port, reference_output

    import shutil

    def make(root, dst):
        script = str(tmp_path / "reference_train.py")
        shutil.copy(os.path.join(root, "train.py"), script)
        json.dump(_losses(script, find_free_port(), str(tmp_path)), open(dst, "w"))

    theirs = json.load(open(reference_output("dropin_train_losses.json", make)))
    ours = _losses(os.path.join(ROOT, "train.py"), find_free_port(), str(tmp_path))
    assert len(theirs) == len(ours) == 20
    assert theirs[-1] < 1.5 < theirs[0]
    assert all(abs(a - b) < 1e-4 for a, b in zip(theirs, ours)), (theirs, ours)
