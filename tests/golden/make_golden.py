"""Generate tests/golden/*.npz by running the UNMODIFIED reference
(/root/reference, sphinxteam/tramp) on seeded inputs.

Run in the build container only (the GPU box has no /root/reference):

    python tests/golden/make_golden.py

The reference is imported through tests/golden/_refshim.py (networkx-1.x veneer
+ matplotlib stub); no reference source is modified or copied.  The outputs are
small fixtures committed to the repo; the oracle (oracle/tramp_oracle.py) and
the CUDA path are both checked against them.
"""
import os
import sys
import logging
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
import _refshim  # noqa: E402

_refshim.install()
logging.disable(logging.CRITICAL)

from tramp.priors import GaussBernoulliPrior, BinaryPrior, GaussianPrior  # noqa: E402
from tramp.likelihoods import GaussianLikelihood, SgnLikelihood, AbsLikelihood  # noqa: E402
from tramp.channels import LinearChannel  # noqa: E402
from tramp.beliefs import truncated, positive, sparse, binary, normal  # noqa: E402
from tramp.variables import SISOVariable as V  # noqa: E402
from tramp.algos import (  # noqa: E402
    ExpectationPropagation, TrackErrors, TrackEvolution, JoinCallback,
    EarlyStoppingEP, ConstantInit, NoisyInit, CustomInit,
)
from tramp.base import Variable  # noqa: E402


def _prior_from(spec):
    kind = spec["kind"]
    kw = {k: v for k, v in spec.items() if k != "kind"}
    return dict(gauss_bernoulli=GaussBernoulliPrior, binary=BinaryPrior,
                gaussian=GaussianPrior)[kind](**kw)


def _lik_from(spec, y):
    kind = spec["kind"]
    kw = {k: v for k, v in spec.items() if k != "kind"}
    return dict(gaussian=GaussianLikelihood, sgn=SgnLikelihood,
                abs=AbsLikelihood)[kind](y=y, **kw)


# --------------------------------------------------------------------------
# A. elementwise factors
# --------------------------------------------------------------------------
from make_golden_specs import PRIOR_SPECS, LIK_SPECS, TRUNC_CASES  # noqa: E402


def _grid():
    """(a, b) grid: the reference's own test inputs (tests/test_priors.py:32-35)
    followed by a stress grid over many decades of precision."""
    n = 100
    a1 = np.linspace(1, 2, n)
    b1 = np.linspace(-2, 2, n)
    a_dec = np.array([1e-11, 1e-6, 1e-3, 0.1, 1.0, 7.0, 1e3, 1e6, 1e11])
    b_lin = np.array([-60., -20., -6., -1.5, -0.3, -1e-3, 0., 1e-3, 0.3, 1.5, 6., 20., 60.])
    A, B = np.meshgrid(a_dec, b_lin, indexing="ij")
    # scale b with sqrt(a) so the stress grid stays in the numerically
    # meaningful region |b|/sqrt(a) <= 60
    a2 = A.ravel()
    b2 = (B * np.sqrt(A)).ravel()
    return np.concatenate([a1, a2]), np.concatenate([b1, b2])


def gen_elementwise(out):
    a, b = _grid()
    n = a.size
    out["grid_a"] = a
    out["grid_b"] = b
    bnorm = b / np.sqrt(a)
    out["grid_bnorm"] = bnorm
    rng = np.random.RandomState(7)
    z = np.concatenate([np.linspace(-3, 3, 100), rng.randn(n - 100) * 2])
    out["grid_z"] = z
    for i, spec in enumerate(PRIOR_SPECS):
        p = _prior_from(dict(spec, size=n, isotropic=False))
        r, v = p.compute_forward_posterior(a, b)
        out[f"prior{i}_r"] = r
        out[f"prior{i}_v"] = v * np.ones(n)
        out[f"prior{i}_A"] = p.scalar_log_partition(a, b)
        # isotropic, scalar a, several precisions
        p_iso = _prior_from(dict(spec, size=n, isotropic=True))
        for j, a_s in enumerate([1e-3, 0.7, 30.0]):
            bb = bnorm * np.sqrt(a_s)      # keep |b|/sqrt(a) <= 60 for the scalar precision too
            r, v = p_iso.compute_forward_posterior(a_s, bb)
            an, bn = p_iso.compute_forward_message(a_s, bb)
            out[f"prior{i}_iso{j}_r"] = r
            out[f"prior{i}_iso{j}_v"] = np.float64(v)
            out[f"prior{i}_iso{j}_anew"] = np.float64(an)
            out[f"prior{i}_iso{j}_bnew"] = bn * np.ones(n)
            out[f"prior{i}_iso{j}_A"] = np.float64(p_iso.compute_log_partition(a_s, bb))
    out["iso_a"] = np.array([1e-3, 0.7, 30.0])
    for i, spec in enumerate(LIK_SPECS):
        y = dict(gaussian=z, sgn=np.sign(z), abs=np.abs(z))[spec["kind"]]
        out[f"lik{i}_y"] = y
        lk = _lik_from(dict(spec, isotropic=False), y)
        r, v = lk.compute_backward_posterior(a, b, y)
        out[f"lik{i}_r"] = r
        out[f"lik{i}_v"] = v * np.ones(n)
        out[f"lik{i}_A"] = lk.scalar_log_partition(a, b, y)
        lk_iso = _lik_from(dict(spec, isotropic=True), y)
        for j, a_s in enumerate([1e-3, 0.7, 30.0]):
            bb = bnorm * np.sqrt(a_s)
            r, v = lk_iso.compute_backward_posterior(a_s, bb, y)
            an, bn = lk_iso.compute_backward_message(a_s, bb)
            out[f"lik{i}_iso{j}_r"] = r
            out[f"lik{i}_iso{j}_v"] = np.float64(v)
            out[f"lik{i}_iso{j}_anew"] = np.float64(an)
            out[f"lik{i}_iso{j}_bnew"] = bn * np.ones(n)
            out[f"lik{i}_iso{j}_A"] = np.float64(lk_iso.compute_log_partition(a_s, bb, y))


def gen_truncated(out):
    b = np.linspace(-6, 6, 121)
    out["trunc_b"] = b
    out["trunc_cases"] = np.array(TRUNC_CASES, dtype=float)
    for i, (a, lo, hi) in enumerate(TRUNC_CASES):
        out[f"trunc{i}_A"] = truncated.A(a, b, lo, hi)
        out[f"trunc{i}_r"] = truncated.r(a, b, lo, hi)
        out[f"trunc{i}_v"] = truncated.v(a, b, lo, hi)
        out[f"trunc{i}_p"] = truncated.p(a, b, lo, hi)
    a = np.array([0.3, 1.0, 4.0])[:, None]
    bb = np.linspace(-40, 40, 161)[None, :]
    out["pos_a"] = a
    out["pos_b"] = bb
    out["pos_A"] = positive.A(a, bb)
    out["pos_r"] = positive.r(a, bb)
    out["pos_v"] = positive.v(a, bb)


def gen_beliefs(out):
    """Every function of tramp/beliefs/{sparse,binary,positive,truncated}.py on grids that
    reach the small-weight regime of the sparse belief (p down to 1e-18)."""
    a = np.array([0.5, 1.0, 3.0, 40.0])[:, None]
    b = np.linspace(-9, 9, 73)[None, :]
    out["bel_a"], out["bel_b"] = a, b
    etas = np.array([-3.0, 0.4, 2.2, 8.0, 15.0, 22.0, 30.0, 40.0])
    out["sparse_eta"] = etas
    for k, eta in enumerate(etas):
        for name in ("A", "p", "r", "v", "tau"):
            out[f"sparse{k}_{name}"] = getattr(sparse, name)(a, b, eta)
    bb = np.linspace(-45, 45, 181)
    out["binary_b"] = bb
    for name in ("A", "r", "v"):
        out[f"binary_{name}"] = getattr(binary, name)(bb)
    for name in ("A", "r", "v", "tau", "p"):
        out[f"positive_{name}"] = getattr(positive, name)(a, b)
    for i, (a_t, lo, hi) in enumerate(TRUNC_CASES):
        bt = out_trunc_b()
        out[f"trunc{i}_tau"] = truncated.tau(a_t, bt, lo, hi)
        out[f"trunc{i}_p"] = truncated.p(a_t, bt, lo, hi)
    out["trunc_b"] = out_trunc_b()
    out["trunc_cases"] = np.array(TRUNC_CASES, dtype=float)


def out_trunc_b():
    return np.linspace(-6, 6, 121)


# --------------------------------------------------------------------------
# B. LinearChannel
# --------------------------------------------------------------------------
def gen_linear(out):
    rng = np.random.RandomState(11)
    Ws = [
        rng.randn(12, 20) / np.sqrt(20),
        rng.randn(20, 12) / np.sqrt(12),
        rng.randn(16, 16) / np.sqrt(16),
        (rng.randn(10, 6) @ rng.randn(6, 16)) / 4.0,    # rank 6 < min(M, N)
    ]
    ab = [(1.0, 2.0), (0.3, 0.0), (1e-11, 5.0), (4.0, 1e-11), (1e3, 1e-3), (0.0, 1.0)]
    out["lin_ab"] = np.array(ab)
    out["lin_nW"] = np.int64(len(Ws))
    for i, W in enumerate(Ws):
        ch = LinearChannel(W)
        M, N = W.shape
        out[f"lin{i}_W"] = W
        out[f"lin{i}_rank"] = np.int64(ch.rank)
        bz = rng.randn(N)
        bx = rng.randn(M)
        out[f"lin{i}_bz"] = bz
        out[f"lin{i}_bx"] = bx
        for j, (az, ax) in enumerate(ab):
            with np.errstate(all="ignore"):
                rz, vz = ch.compute_backward_posterior(az, bz, ax, bx)
                rx, vx = ch.compute_forward_posterior(az, bz, ax, bx) if az > 0 else (np.full(M, np.nan), np.nan)
                A = ch.compute_log_partition(az, bz, ax, bx)
            out[f"lin{i}_{j}_rz"] = rz
            out[f"lin{i}_{j}_vz"] = np.float64(vz)
            out[f"lin{i}_{j}_rx"] = rx
            out[f"lin{i}_{j}_vx"] = np.float64(vx)
            out[f"lin{i}_{j}_A"] = np.float64(A)
            out[f"lin{i}_{j}_neff"] = np.float64(ch.compute_n_eff(az, ax))


# --------------------------------------------------------------------------
# C. EP sweeps through the unmodified driver
# --------------------------------------------------------------------------
class _Never:
    """A callback that records and never stops (fixed iteration count)."""

    def __init__(self, x_true):
        self.x_true = x_true
        self.mse, self.vx, self.vz = [], [], []

    def __call__(self, algo, i, max_iter):
        d = algo.get_variables_data()
        self.mse.append(np.mean((d["x"]["r"] - self.x_true)**2))
        self.vx.append(float(d["x"]["v"]))
        self.vz.append(float(d["z"]["v"]))


SWEEPS = [
    # name, N, M, prior, lik, damping, n_iter, seed, init
    dict(name="cs_gb_gauss", N=200, M=100, prior=dict(kind="gauss_bernoulli", rho=0.1),
         lik=dict(kind="gaussian", var=1e-2), damping=None, n_iter=40, seed=42),
    dict(name="cs_gb_gauss_damped", N=128, M=64, prior=dict(kind="gauss_bernoulli", rho=0.1),
         lik=dict(kind="gaussian", var=1e-2), damping=0.5, n_iter=40, seed=43),
    dict(name="perceptron_gauss_sgn", N=100, M=200, prior=dict(kind="gaussian"),
         lik=dict(kind="sgn"), damping=0.5, n_iter=30, seed=44),
    dict(name="binary_sgn", N=96, M=160, prior=dict(kind="binary", p_pos=0.5),
         lik=dict(kind="sgn"), damping=0.3, n_iter=30, seed=45),
    dict(name="phase_binary_abs", N=96, M=192, prior=dict(kind="binary", p_pos=0.6),
         lik=dict(kind="abs"), damping=0.3, n_iter=40, seed=46),
    dict(name="gb_sgn_damped", N=150, M=150, prior=dict(kind="gauss_bernoulli", rho=0.3),
         lik=dict(kind="sgn"), damping=0.2, n_iter=30, seed=47),
    dict(name="gb_abs_noisyinit", N=100, M=130, prior=dict(kind="gauss_bernoulli", rho=0.5),
         lik=dict(kind="abs"), damping=0.3, n_iter=30, seed=48, init="noisy"),
    dict(name="cs_noiseless", N=120, M=90, prior=dict(kind="gauss_bernoulli", rho=0.1),
         lik=dict(kind="gaussian", var=1e-10), damping=None, n_iter=40, seed=49),
    dict(name="cs_odd_shape", N=77, M=33, prior=dict(kind="gauss_bernoulli", rho=0.2, mean=0.5, var=2.0),
         lik=dict(kind="gaussian", var=0.05), damping=0.1, n_iter=25, seed=50),
]


def _sample_prior(spec, N):
    return _prior_from(dict(spec, size=N)).sample()


def _observe(kind, z, var, rng_noise):
    if kind == "gaussian":
        return z + np.sqrt(var) * rng_noise
    if kind == "sgn":
        return np.where(z >= 0, 1.0, -1.0)   # SgnChannel.sample: +1 at z == 0
    if kind == "abs":
        return np.abs(z)
    raise ValueError(kind)


def run_sweep(cfg, out, early=False):
    name = cfg["name"] + ("_early" if early else "")
    N, M = cfg["N"], cfg["M"]
    np.random.seed(cfg["seed"])
    W = np.random.randn(M, N) / np.sqrt(N)            # GaussianEnsemble.generate
    x = _sample_prior(cfg["prior"], N).astype(float)
    z = W @ x
    y = _observe(cfg["lik"]["kind"], z, cfg["lik"].get("var", 1), np.random.standard_normal(M))
    prior = _prior_from(dict(cfg["prior"], size=N))
    lik = _lik_from(cfg["lik"], y)
    model = (prior @ V("x") @ LinearChannel(W) @ V("z") @ lik).to_model()
    ep = ExpectationPropagation(model)
    init = None
    if cfg.get("init") == "noisy":
        np.random.seed(cfg["seed"] + 1000)
        init = NoisyInit(a_mean=0.5, a_var=0, b_mean=0, b_var=0.25)
    if early:
        ep.iterate(max_iter=200, callback=EarlyStoppingEP(), initializer=init,
                   damping=cfg["damping"])
    else:
        cb = _Never(x)
        if init is not None:
            # record the initial messages NoisyInit drew: init_message_dag is
            # called inside iterate(), so rerun it by hand first to capture them
            np.random.seed(cfg["seed"] + 1000)
            ep.init_message_dag(init)
            _dump_edges(ep, out, name + "_init")
            np.random.seed(cfg["seed"] + 1000)
        ep.iterate(max_iter=cfg["n_iter"], callback=cb, initializer=init,
                   damping=cfg["damping"])
        out[name + "_mse"] = np.array(cb.mse)
        out[name + "_vx"] = np.array(cb.vx)
        out[name + "_vz"] = np.array(cb.vz)
    d = ep.get_variables_data()
    out[name + "_W"] = W
    out[name + "_y"] = y
    out[name + "_x"] = x
    out[name + "_rx"] = d["x"]["r"]
    out[name + "_rz"] = d["z"]["r"]
    out[name + "_vx_final"] = np.float64(d["x"]["v"])
    out[name + "_vz_final"] = np.float64(d["z"]["v"])
    out[name + "_n_iter"] = np.int64(ep.n_iter)
    _dump_edges(ep, out, name)
    out[name + "_logZ"] = np.float64(ep.log_evidence())
    for node, data in ep.message_dag.nodes(data=True):
        tag = node.id if isinstance(node, Variable) else type(node).__name__
        out[name + "_A_" + tag] = np.float64(data["A"])


def run_diverging(out):
    """An instance on which the default EarlyStoppingEP takes its `max_increase`
    branch (callbacks.py:275-283): restore the previous iteration and stop."""
    name = "cs_diverges_early"
    rng = np.random.RandomState(9)
    B, N, M = 4, 120, 60
    W = rng.randn(B, M, N) / np.sqrt(N)
    x = rng.randn(B, N) * (rng.rand(B, N) < 0.1)
    y = np.einsum("bmn,bn->bm", W, x) + 0.1 * rng.randn(B, M)
    W, x, y = W[3], x[3], y[3]
    model = (GaussBernoulliPrior(size=N, rho=0.1) @ V("x") @ LinearChannel(W) @ V("z")
             @ GaussianLikelihood(y=y, var=1e-2)).to_model()
    ep = ExpectationPropagation(model)
    ep.iterate(max_iter=200)
    d = ep.get_variables_data()
    out[name + "_W"], out[name + "_y"], out[name + "_x"] = W, y, x
    out[name + "_rx"], out[name + "_rz"] = d["x"]["r"], d["z"]["r"]
    out[name + "_vx_final"], out[name + "_vz_final"] = np.float64(d["x"]["v"]), np.float64(d["z"]["v"])
    out[name + "_n_iter"] = np.int64(ep.n_iter)
    _dump_edges(ep, out, name)


# --------------------------------------------------------------------------
# D. adaptive damping (message_passing.py:151-185), update_dA (:129-149),
#    TrackObjective (callbacks.py:63-85)
# --------------------------------------------------------------------------
ADAPTIVE = [
    dict(name="ad_gb_sgn", N=60, M=80, prior=dict(kind="gauss_bernoulli", rho=0.3), lik=dict(kind="sgn"),
         damping="adaptive", update_dA=False, n_iter=8, seed=61),
    dict(name="ad_gb_gauss", N=64, M=32, prior=dict(kind="gauss_bernoulli", rho=0.1),
         lik=dict(kind="gaussian", var=1e-2), damping="adaptive", update_dA=False, n_iter=8, seed=62),
    dict(name="dA_gb_sgn", N=60, M=80, prior=dict(kind="gauss_bernoulli", rho=0.3), lik=dict(kind="sgn"),
         damping=0.2, update_dA=True, n_iter=8, seed=63),
    dict(name="dA_gauss_sgn", N=48, M=96, prior=dict(kind="gaussian"), lik=dict(kind="sgn"),
         damping=None, update_dA=True, n_iter=6, seed=64),
]


class _Objective:
    def __init__(self, x_true):
        self.x_true, self.mse, self.vx, self.vz, self.A = x_true, [], [], [], []

    def __call__(self, algo, i, max_iter):
        d = algo.get_variables_data()
        self.mse.append(np.mean((d["x"]["r"] - self.x_true)**2))
        self.vx.append(float(d["x"]["v"]))
        self.vz.append(float(d["z"]["v"]))
        algo.update_objective()
        self.A.append(float(algo.A_model))


def run_adaptive(cfg, out):
    name, N, M = cfg["name"], cfg["N"], cfg["M"]
    np.random.seed(cfg["seed"])
    W = np.random.randn(M, N) / np.sqrt(N)
    x = _sample_prior(cfg["prior"], N).astype(float)
    y = _observe(cfg["lik"]["kind"], W @ x, cfg["lik"].get("var", 1), np.random.standard_normal(M))
    model = (_prior_from(dict(cfg["prior"], size=N)) @ V("x") @ LinearChannel(W) @ V("z")
             @ _lik_from(cfg["lik"], y)).to_model()
    ep = ExpectationPropagation(model)
    cb = _Objective(x)
    ep.iterate(max_iter=cfg["n_iter"], callback=cb, damping=cfg["damping"], update_dA=cfg["update_dA"])
    out[name + "_W"], out[name + "_y"], out[name + "_x"] = W, y, x
    out[name + "_mse"], out[name + "_vx"], out[name + "_vz"] = np.array(cb.mse), np.array(cb.vx), np.array(cb.vz)
    out[name + "_A_model"] = np.array(cb.A)
    d = ep.get_variables_data()
    out[name + "_rx"], out[name + "_rz"] = d["x"]["r"], d["z"]["r"]
    _dump_edges(ep, out, name, extra=("dA", "beta", "n_iter"))


def _dump_edges(ep, out, name, extra=()):
    """Store the 8 edges under the SURVEY 3.3 names e1..e8."""
    for s, t, data in ep.message_dag.edges(data=True):
        var = s if isinstance(s, Variable) else t
        fac = t if isinstance(s, Variable) else s
        fname = type(fac).__name__
        d = data["direction"]
        if var.id == "x":
            if "Prior" in fname:
                e = "e1" if d == "fwd" else "e8"
            else:
                e = "e2" if d == "fwd" else "e7"
        else:
            if "Linear" in fname:
                e = "e3" if d == "fwd" else "e6"
            else:
                e = "e4" if d == "fwd" else "e5"
        out[f"{name}_{e}_a"] = np.float64(data["a"])
        out[f"{name}_{e}_b"] = np.asarray(data["b"], dtype=float) * np.ones(
            ep.model_dag.node[var]["shape"])
        for key in extra:
            val = data.get(key)
            out[f"{name}_{e}_{key}"] = np.float64(np.nan if val is None else val)


def main():
    el = {}
    gen_elementwise(el)
    gen_truncated(el)
    np.savez_compressed(os.path.join(HERE, "elementwise.npz"), **el)
    bel = {}
    with np.errstate(all="ignore"):
        gen_beliefs(bel)
    np.savez_compressed(os.path.join(HERE, "beliefs.npz"), **bel)
    lin = {}
    gen_linear(lin)
    np.savez_compressed(os.path.join(HERE, "linear.npz"), **lin)
    sw = {}
    for cfg in SWEEPS:
        with np.errstate(all="ignore"):
            run_sweep(cfg, sw)
    for cfg in SWEEPS[:3]:
        run_sweep(cfg, sw, early=True)
    run_diverging(sw)
    import hashlib
    import json
    sw["configs"] = np.array(json.dumps(SWEEPS))
    # W is most of the file and is redrawn from its seed by tests.golden.load_sweeps: store its digest
    sw = {(k + "_sha256" if k.endswith("_W") else k):
          (np.array(hashlib.sha256(v.tobytes()).hexdigest()) if k.endswith("_W") else v) for k, v in sw.items()}
    np.savez_compressed(os.path.join(HERE, "sweeps.npz"), **sw)
    ad = {}
    for cfg in ADAPTIVE:
        with np.errstate(all="ignore"):
            run_adaptive(cfg, ad)
    ad["configs"] = np.array(json.dumps(ADAPTIVE))
    np.savez_compressed(os.path.join(HERE, "adaptive.npz"), **ad)
    for f in ("elementwise.npz", "beliefs.npz", "linear.npz", "sweeps.npz", "adaptive.npz"):
        print(f, os.path.getsize(os.path.join(HERE, f)) // 1024, "KiB")


if __name__ == "__main__":
    main()
