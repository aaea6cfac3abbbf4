"""Generate tests/golden/train/trajectories.npz from the UNMODIFIED reference (test infrastructure).

Run where a checkout of the reference project is available (read-only):

    DSMIL_REFERENCE=<reference checkout> python oracle/gen_train_golden.py

Trains the reference's own MILNet(FCLayer, BClassifier) on CPU fp32 with tests/helpers.train_trajectory on the
seeded datasets of tests/helpers.training_case and stores the loss of every training step and every held-out bag.
tests/test_zz_acceptance_gpu.py trains this repo's MILNet the same way on the GPU and compares.  Inputs are not
stored: a CRC of the regenerated bags detects RNG drift.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from oracle.gen_golden import build_ref_model, load_reference  # noqa: E402
import helpers  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "train")


def main():
    os.makedirs(OUT, exist_ok=True)
    ref = load_reference()
    torch.set_num_threads(1)  # fixed reduction order for the stored fp32 losses
    out = {}
    for name in helpers.TRAINING_CASES:
        p, bags, _ = helpers.training_case(name)
        net = build_ref_model(ref, p).train()
        out[name] = helpers.train_trajectory(net, name, "cpu")
        out[name + "_x_crc"] = helpers.bags_crc(bags)
        print(name, out[name].shape, out[name][:, :4])
    np.savez_compressed(os.path.join(OUT, "trajectories.npz"), **out)


if __name__ == "__main__":
    main()
