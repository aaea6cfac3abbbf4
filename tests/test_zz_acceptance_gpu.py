"""Acceptance harness (SURVEY §8(b)): the reference's own training drivers, UNMODIFIED, run against this repo's
`dsmil` shim on the device -- and, on the same seeds, against the reference's own `dsmil.py` through PyTorch eager
on the same GPU.  The two runs must print the same loss trajectory.

The drivers are staged byte-for-byte into the git-ignored `oracle/_ref/` by `__graft_entry__.build()` when the
reference checkout is present (oracle/stage_ref.py); the reference checkout is never read at run time.  Without
them those tests skip, and `test_training_matches_reference` stands in: it trains this repo's MILNet on bags of
the drivers' shapes and compares every loss with the reference MILNet's, stored in tests/golden/train/.

    train_tcga.py:199-429   5-fold CV over `.pt` bags built from `datasets/<name>/<name>.csv`  (D=512, C=2)
    train_mil.py:112-187    classic MIL (musk1: D=166, C=1), 3 folds
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import stage_ref  # noqa: E402
from helpers import TRAINING_CASES, bags_crc, build_net, train_trajectory, training_case  # noqa: E402

pytestmark = pytest.mark.gpu
RUNNER = os.path.join(ROOT, "tests", "run_reference_caller.py")


def _run(which, script, args, cwd):
    env = dict(os.environ)
    env.pop("PYTHONPATH", None)
    r = subprocess.run([sys.executable, RUNNER, which, script, *args], cwd=cwd, env=env, capture_output=True,
                       text=True, timeout=600)
    assert r.returncode == 0, f"{script} ({which}) failed:\n{r.stdout[-3000:]}\n{r.stderr[-3000:]}"
    return r.stdout


def _need_ref(name):
    if stage_ref.staged(name) is None or stage_ref.staged("dsmil.py") is None:
        pytest.skip("reference sources not staged in oracle/_ref (__graft_entry__.build() stages them from a reference "
                    "checkout, see oracle/stage_ref.py)")


def test_staged_reference_is_unmodified():
    import hashlib
    import json
    _need_ref("dsmil.py")
    man = json.load(open(os.path.join(stage_ref.REF_DST, "MANIFEST.json")))["sha256"]
    for f, h in man.items():
        assert hashlib.sha256(open(os.path.join(stage_ref.REF_DST, f), "rb").read()).hexdigest() == h, f


def test_train_tcga_unmodified(tmp_path):
    """train_tcga.py, one epoch x 5 folds on a synthetic two-class dataset written in the reference's wire format."""
    _need_ref("train_tcga.py")
    from dsmil_wsi_b200 import embed, formats
    rng = np.random.default_rng(7)
    ds = tmp_path / "datasets" / "synth"
    for cls in ("0_luad", "1_lusc"):
        for b in range(40):       # 16-bag test folds: every fold holds both classes (an all-one-class fold makes the
            n = int(rng.integers(60, 160))   # reference's own AUC bookkeeping fail, train_tcga.py:290)
            x = rng.random((n, 512), dtype=np.float32)
            if cls.startswith("1"):
                x[: n // 8, :32] += 1.5        # a few "tumour" patches carry the class signal
            embed.write_bag_csv(x, str(ds), os.path.join(str(ds), cls, f"{cls}_bag{b}"))
    # index paths must be relative to the cwd the driver runs in (train_tcga.py:245-250 reads them as given)
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        formats.write_dataset_index(os.path.join("datasets", "synth"), "synth", rng=np.random.default_rng(1))
    finally:
        os.chdir(cwd)
    args = ["--dataset", "synth", "--num_epochs", "1", "--num_classes", "2", "--feats_size", "512"]
    ours = _run("ours", "train_tcga.py", args, str(tmp_path))
    assert "DSMIL_MODULE=" + os.path.join(ROOT, "dsmil.py") in ours
    launches = int(re.search(r"DSMIL_LAUNCHES=(\d+)", ours).group(1))
    assert launches > 100, "the unmodified driver did not run on libdsmil_b200.so"
    pat = re.compile(r"Epoch \[1/1\] train loss: ([0-9.]+) test loss: ([0-9.]+)")
    l_ours = [(float(a), float(b)) for a, b in pat.findall(ours)]
    assert len(l_ours) == 5, ours[-2000:]
    ref = _run("ref", "train_tcga.py", args, str(tmp_path))
    assert "DSMIL_MODULE=" + os.path.join(ROOT, "oracle", "_ref", "dsmil.py") in ref
    l_ref = [(float(a), float(b)) for a, b in pat.findall(ref)]
    assert len(l_ref) == 5
    # 4 printed decimals; one epoch of Adam steps on 64 bags: identical up to the last printed digit or two
    assert np.allclose(np.array(l_ours), np.array(l_ref), atol=3e-4), (l_ours, l_ref)


def test_train_mil_unmodified(tmp_path):
    """train_mil.py (classic MIL, D=166, C=1) on a synthetic musk1-shaped file, 2 epochs x 3 folds."""
    _need_ref("train_mil.py")
    from dsmil_wsi_b200 import formats
    rng = np.random.default_rng(3)
    bags = []
    for b in range(30):
        n = int(rng.integers(3, 12))
        x = rng.standard_normal((n, 166)).astype(np.float32)
        label = b % 2
        if label:
            x[0, :8] += 2.0
        bags.append((label, x))
    d = tmp_path / "datasets" / "mil_dataset" / "Musk"
    d.mkdir(parents=True)
    formats.write_mil_svm(str(d / "musk1norm.svm"), bags)
    args = ["--datasets", "musk1", "--num_epoch", "2", "--cv_fold", "3"]
    ours = _run("ours", "train_mil.py", args, str(tmp_path))
    assert "DSMIL_MODULE=" + os.path.join(ROOT, "dsmil.py") in ours
    assert int(re.search(r"DSMIL_LAUNCHES=(\d+)", ours).group(1)) > 100
    pat = re.compile(r"Epoch \[2/2\] train loss: ([0-9.]+), test loss: ([0-9.]+)")
    l_ours = [(float(a), float(b)) for a, b in pat.findall(ours)]
    assert len(l_ours) == 3, ours[-2000:]
    ref = _run("ref", "train_mil.py", args, str(tmp_path))
    l_ref = [(float(a), float(b)) for a, b in pat.findall(ref)]
    assert len(l_ref) == 3
    assert np.allclose(np.array(l_ours), np.array(l_ref), atol=3e-4), (l_ours, l_ref)


@pytest.mark.parametrize("name", sorted(TRAINING_CASES))
def test_training_matches_reference(name):
    """Two-class training on bags of train_tcga.py's / train_mil.py's shape: this repo's MILNet on the device and the
    reference's MILNet (torch-CPU fp32, oracle/gen_train_golden.py), same weights, same bag order, same loss and Adam:
    the loss of every step and every held-out bag agrees."""
    from dsmil_wsi_b200 import _lib
    g = np.load(os.path.join(ROOT, "tests", "golden", "train", "trajectories.npz"))
    p, bags, _ = training_case(name)
    assert bags_crc(bags) == g[name + "_x_crc"], "numpy RNG stream drifted (bags)"
    n0 = _lib.launch_count()
    losses = train_trajectory(build_net(p, "cuda"), name, "cuda")
    assert _lib.launch_count() - n0 > 100, "training did not run on libdsmil_b200.so"
    assert losses.shape == g[name].shape
    assert np.allclose(losses, g[name], rtol=0, atol=3e-4), np.abs(losses - g[name]).max()
