import hashlib
import json
import os

import numpy as np


def _sweep_operator(name, cfgs):
    """The matrix W of golden run `name`, drawn as tests/golden/make_golden.py drew it."""
    if name == "cs_diverges_early":                     # run_diverging: instance 3 of a batch of 4
        return (np.random.RandomState(9).randn(4, 60, 120) / np.sqrt(120))[3]
    cfg = cfgs[name[:-len("_early")] if name.endswith("_early") else name]      # run_sweep
    return np.random.RandomState(cfg["seed"]).randn(cfg["M"], cfg["N"]) / np.sqrt(cfg["N"])


def load_sweeps(golden_dir):
    """sweeps.npz as a dict, with the W of every run put back.

    The file stores the SHA-256 of each W instead of W itself (random float64 does not
    compress, and the matrices would be most of the file); W is redrawn from the run's
    seed and must hash to the stored digest, so the tests see exactly the operators the
    reference ran on."""
    with np.load(os.path.join(golden_dir, "sweeps.npz")) as f:
        sw = {k: f[k] for k in f.files}
    cfgs = {c["name"]: c for c in json.loads(str(sw["configs"]))}
    for key in [k for k in sw if k.endswith("_W_sha256")]:
        name = key[:-len("_W_sha256")]
        W = _sweep_operator(name, cfgs)
        assert hashlib.sha256(W.tobytes()).hexdigest() == str(sw[key]), f"redrawn W of {name} differs"
        sw[name + "_W"] = W
    return sw
