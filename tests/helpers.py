"""Test helpers (test infrastructure; may use oracle/)."""
import ctypes
import zlib

import numpy as np
import torch

from oracle import dsmil_oracle as orc


def state_dict_from_params(p: orc.Params, iclassifier=False):
    t = lambda a: torch.from_numpy(np.array(a, dtype=np.float32))
    ik = "i_classifier.fc." if iclassifier else "i_classifier.fc.0."
    sd = {ik + "weight": t(p.Wi), ik + "bias": t(p.bi),
          "b_classifier.fcc.weight": t(p.Wf), "b_classifier.fcc.bias": t(p.bf)}
    if p.nonlinear:
        sd.update({"b_classifier.q.0.weight": t(p.W1), "b_classifier.q.0.bias": t(p.b1),
                   "b_classifier.q.2.weight": t(p.W2), "b_classifier.q.2.bias": t(p.b2)})
    else:
        sd.update({"b_classifier.q.weight": t(p.W1), "b_classifier.q.bias": t(p.b1)})
    if p.passing_v:
        sd.update({"b_classifier.v.1.weight": t(p.Wv), "b_classifier.v.1.bias": t(p.bv)})
    return sd


def build_net(p: orc.Params, device="cuda", dropout_v=0.0):
    import dsmil as mil
    net = mil.MILNet(mil.FCLayer(p.D, p.C),
                     mil.BClassifier(p.D, p.C, dropout_v=dropout_v, nonlinear=p.nonlinear, passing_v=p.passing_v))
    net.load_state_dict(state_dict_from_params(p), strict=True)
    return net.to(device)


def caller_loss(classes, pred, y):
    """train_tcga.py:67-71"""
    crit = torch.nn.BCEWithLogitsLoss()
    mx, _ = torch.max(classes, 0)
    return 0.5 * crit(pred.view(1, -1), y.view(1, -1)) + 0.5 * crit(mx.view(1, -1), y.view(1, -1))


GRAD_MAP = {"Wi": "i_classifier.fc.0.weight", "bi": "i_classifier.fc.0.bias",
            "Wf": "b_classifier.fcc.weight", "bf": "b_classifier.fcc.bias",
            "Wv": "b_classifier.v.1.weight", "bv": "b_classifier.v.1.bias"}


def grad_name(short, nonlinear):
    if short in GRAD_MAP:
        return GRAD_MAP[short]
    if nonlinear:
        return {"W1": "b_classifier.q.0.weight", "b1": "b_classifier.q.0.bias",
                "W2": "b_classifier.q.2.weight", "b2": "b_classifier.q.2.bias"}[short]
    return {"W1": "b_classifier.q.weight", "b1": "b_classifier.q.bias"}[short]


def pred_tolerance_ok(pred, ref_pred, p: orc.Params, B_ref, tol):
    """|d| <= tol * max(|logit|, scale of the GEMV terms): the fcc GEMV cancels (SURVEY §7.2-2)."""
    terms = np.abs(p.Wf.reshape(p.C, -1)).astype(np.float64) @ np.abs(np.asarray(B_ref, np.float64).reshape(-1))
    err = np.abs(np.asarray(pred, np.float64).reshape(-1) - np.asarray(ref_pred, np.float64).reshape(-1))
    return bool(np.all(err <= tol * np.maximum(np.abs(np.asarray(ref_pred, np.float64).reshape(-1)), terms))), err


def scores_close(a, b, tol=2e-6):
    """Instance scores from two DIFFERENT kernels (pair kernel / k_qmlp_sm100 / k_scores: each sums the D products of a
    row in its own fixed order): equal to the tolerance every path is held to against the reference (2e-6 of the
    largest score); the arg-max they select is asserted bit-exact separately."""
    a = a.detach().float().cpu().numpy().astype(np.float64)
    b = b.detach().float().cpu().numpy().astype(np.float64)
    return a.shape == b.shape and float(np.max(np.abs(a - b))) <= tol * max(float(np.max(np.abs(b))), 1e-30)


# name: (D, C, wseed, dataseed, train bags, test bags, epochs).  "tcga" has train_tcga.py's shape (D=512, C=2,
# 60-159 patches per bag), "musk" train_mil.py's (musk1: D=166, C=1, 3-11 instances per bag).
TRAINING_CASES = {"tcga": (512, 2, 201, 7, 16, 8, 2), "musk": (166, 1, 202, 3, 20, 10, 3)}


def training_case(name):
    """(Params, bags, labels) of a seeded two-class synthetic dataset; a few instances of each bag carry its class."""
    D, C, wseed, dseed, n_train, n_test, _ = TRAINING_CASES[name]
    p = orc.random_params(D, C, wseed)
    rng = np.random.default_rng(dseed)
    bags, labels = [], []
    for b in range(n_train + n_test):
        cls = b % 2
        if name == "tcga":
            n = int(rng.integers(60, 160))
            x = rng.random((n, D), dtype=np.float32)
            x[: n // 8, 32 * cls: 32 * cls + 32] += 1.5
            y = np.eye(C, dtype=np.float32)[cls]
        else:
            n = int(rng.integers(3, 12))
            x = rng.standard_normal((n, D), dtype=np.float32)
            if cls:
                x[0, :8] += 2.0
            y = np.array([cls], np.float32)
        bags.append(x)
        labels.append(y)
    return p, bags, labels


def bags_crc(bags):
    return np.uint32(zlib.crc32(b"".join(np.ascontiguousarray(x).tobytes() for x in bags)))


def train_trajectory(net, name, device):
    """Trains `net` (holding training_case(name)'s weights) the way the reference's drivers do -- one bag per step,
    0.5 * BCE(bag logits) + 0.5 * BCE(max instance score), Adam(betas=(0.5, 0.9)) as train_tcga.py sets it up -- in
    a seeded bag order, and after every epoch scores the held-out bags in eval mode.  Returns the loss of every
    step and every held-out bag, [epochs, train bags + test bags]."""
    _, bags, labels = training_case(name)
    _, _, _, _, n_train, _, epochs = TRAINING_CASES[name]
    xs = [torch.from_numpy(x).to(device) for x in bags]
    ys = [torch.from_numpy(y).to(device) for y in labels]
    opt = torch.optim.Adam(net.parameters(), lr=2e-4, betas=(0.5, 0.9), weight_decay=5e-3)
    out = []
    for epoch in range(epochs):
        row = []
        net.train()
        for i in np.random.default_rng(epoch).permutation(n_train):
            opt.zero_grad()
            classes, pred, _, _ = net(xs[i])
            loss = caller_loss(classes, pred, ys[i])
            loss.backward()
            opt.step()
            row.append(loss.item())
        net.eval()
        with torch.no_grad():
            for i in range(n_train, len(xs)):
                classes, pred, _, _ = net(xs[i])
                row.append(caller_loss(classes, pred, ys[i]).item())
        out.append(row)
    return np.array(out)
