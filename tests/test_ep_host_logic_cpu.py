"""CPU coverage of the Python side of the EP driver: the public-API calls of
tests/test_gpu_api.py with `trb_sweep_run` emulated by the oracle
(tests/_emulated_device.py).  Under test: model compilation, initialisers and
damping maps into the descriptor, the device-replay and the synchronous callback
paths, chunked early stopping, snapshots / roll-back, scenarios -- not kernels."""
import os
import numpy as np
import pytest
from numpy.testing import assert_allclose

from tests._emulated_device import emulated_device  # noqa: F401  (fixture)
from tests.golden import load_sweeps
from tests.test_gpu_api import _build, _configs, _SeqInit


@pytest.fixture(scope="module")
def sw(golden_dir):
    return load_sweeps(golden_dir)


@pytest.mark.parametrize("idx", [0, 1, 2, 6, 8])
def test_public_api_reproduces_golden_sweeps(emulated_device, sw, idx):  # noqa: F811
    from tramp_b200.algos import ExpectationPropagation, TrackErrors, TrackEvolution, JoinCallback
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, sw, name))
    track, evo = TrackErrors({"x": sw[name + "_x"]}), TrackEvolution()
    init = _SeqInit(sw, name) if cfg.get("init") == "noisy" else None
    ep.iterate(max_iter=cfg["n_iter"], callback=JoinCallback([track, evo]), initializer=init,
               damping=cfg["damping"])
    assert ep.n_iter == cfg["n_iter"] and emulated_device.calls["sweep_iterations"] == cfg["n_iter"]
    mse = np.array([e["mse"] for e in track.errors])
    assert_allclose(mse, sw[name + "_mse"], rtol=1e-9)
    df = evo.get_dataframe()
    assert_allclose(df[df.id == "x"].v.values, sw[name + "_vx"], rtol=1e-9)
    assert_allclose(df[df.id == "z"].v.values, sw[name + "_vz"], rtol=1e-9)
    d = ep.get_variables_data()
    ref = sw[name + "_rx"]
    assert_allclose(d["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    assert d["x"]["r"].shape == (cfg["N"],) and isinstance(d["x"]["v"], float)
    for k in range(1, 9):
        a, b = ep._edge(f"e{k}")
        assert_allclose(a, sw[f"{name}_e{k}_a"], rtol=1e-9)


def test_early_stopping_chunks_and_rollback(emulated_device, sw):  # noqa: F811
    from tramp_b200.algos import ExpectationPropagation, TrackEstimate, JoinCallback, EarlyStoppingEP
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    for idx in range(3):                      # default EarlyStoppingEP, device path in chunks of 16
        cfg = _configs(sw)[idx]
        name = cfg["name"] + "_early"
        ep = ExpectationPropagation(_build(cfg, sw, name))
        ep.iterate(max_iter=200, damping=cfg["damping"])
        assert ep.n_iter == int(sw[name + "_n_iter"])
        ref = sw[name + "_rx"]
        assert_allclose(ep.get_variables_data()["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    name = "cs_diverges_early"                # divergence: rolled back to the previous iteration
    for callback in (None, JoinCallback([TrackEstimate(ids=["x"]), EarlyStoppingEP()])):
        model = (GaussBernoulliPrior(size=120, rho=0.1) @ V("x") @ LinearChannel(sw[name + "_W"])
                 @ V("z") @ GaussianLikelihood(y=sw[name + "_y"], var=1e-2)).to_model()
        ep = ExpectationPropagation(model)
        ep.iterate(max_iter=200, callback=callback)
        assert ep.n_iter == int(sw[name + "_n_iter"]) == 7
        d = ep.get_variables_data()
        assert_allclose(d["x"]["r"], sw[name + "_rx"], rtol=1e-9, atol=1e-12)
        assert_allclose(d["x"]["v"], sw[name + "_vx_final"], rtol=1e-9)


def test_n_iter_per_instance_after_a_callback_stop(emulated_device, sw):  # noqa: F811
    """A stopping callback that is not device-replayable takes the one-launch-per-iteration
    path; its early return must still leave `n_iter_per_instance` describing THIS call (it used
    to keep the previous call's value, which run_ep_sharded then gathered)."""
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    cfg = _configs(sw)[0]
    ep = ExpectationPropagation(_build(cfg, sw, cfg["name"]))
    ep.iterate(max_iter=5, callback=PassCallback())
    assert ep.n_iter_per_instance.tolist() == [5]

    class StopAt:                               # a user callback: synchronous path
        def __call__(self, algo, i, max_iter):
            return i == 7
    ep.iterate(max_iter=100, callback=StopAt())
    assert ep.n_iter == 8 and ep.n_iter_per_instance.tolist() == [8]
    ep.iterate(max_iter=3, callback=StopAt(), warm_start=True)
    assert ep.n_iter == 11 and ep.n_iter_per_instance.tolist() == [11]


def test_warm_start_and_nan(emulated_device, sw):  # noqa: F811
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    cfg = _configs(sw)[0]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, sw, name))
    ep.iterate(max_iter=15, callback=PassCallback())
    ep.iterate(max_iter=cfg["n_iter"] - 15, callback=PassCallback(), warm_start=True)
    assert ep.n_iter == cfg["n_iter"]
    ref = sw[name + "_rx"]
    assert_allclose(ep.get_variables_data()["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    y_bad = sw[name + "_y"].copy()
    y_bad[3] = np.nan
    bad = (GaussBernoulliPrior(size=cfg["N"], rho=0.1) @ V("x") @ LinearChannel(sw[name + "_W"]) @ V("z")
           @ GaussianLikelihood(y=y_bad, var=1e-2)).to_model()
    with pytest.raises(ValueError, match="nan"):
        ExpectationPropagation(bad).iterate(max_iter=3, callback=PassCallback())


def test_scenario_reproduces_the_reference_run(emulated_device):  # noqa: F811
    """BayesOptimalScenario.run_all("EP,SE") with EarlyStopping, seed protocol of the
    reference: the unmodified reference printed SE v = 0.009469020882561508 (14
    iterations), EP v = 0.01149781034627002 (17 iterations), mse = 0.012888367874476584."""
    from tramp_b200.models import glm_generative
    from tramp_b200.experiments import BayesOptimalScenario
    from tramp_b200.algos import EarlyStopping
    np.random.seed(5)
    model = glm_generative(N=400, alpha=0.7, ensemble_type="gaussian", prior_type="gauss_bernoulli",
                           output_type="gaussian", prior_rho=0.2, output_var=1e-2)
    scenario = BayesOptimalScenario(model, x_ids=["x"])
    by = {r["source"]: r for r in scenario.run_all(metrics=["mse"], max_iter=100, callback=EarlyStopping())}
    assert_allclose(by["SE"]["v"], 0.009469020882561508, rtol=1e-8)
    assert_allclose(by["EP"]["v"], 0.01149781034627002, rtol=1e-8)
    assert_allclose(by["mse"]["v"], 0.012888367874476584, rtol=1e-8)
    assert by["SE"]["n_iter"] == 14 and by["EP"]["n_iter"] == 17
    df = scenario.ep_convergence(metrics=["mse"], max_iter=12, damping=0.1)
    assert list(df.columns) == ["id", "iter", "mse", "v"] and len(df) == 12
    assert_allclose(scenario.compute_score(scenario.x_pred)["x"]["mse"], df.mse.values[-1], rtol=1e-9)


def test_belief_wrappers_route_to_the_device_routine(emulated_device, golden_dir):  # noqa: F811
    """beliefs.truncated / beliefs.positive (reference beliefs/truncated.py, positive.py)
    are thin natural-parameter wrappers over one device routine; with that routine
    emulated by the oracle they must reproduce the reference's golden values."""
    from tramp_b200.beliefs import truncated, positive
    g = np.load(os.path.join(golden_dir, "elementwise.npz"))
    b = g["trunc_b"]
    for i, (a, lo, hi) in enumerate(g["trunc_cases"]):
        for key, fn in (("A", truncated.A), ("r", truncated.r), ("v", truncated.v), ("p", truncated.p)):
            assert_allclose(fn(a, b, lo, hi), g[f"trunc{i}_{key}"], rtol=1e-12, atol=1e-300)
        assert_allclose(truncated.tau(a, b, lo, hi), g[f"trunc{i}_r"]**2 + g[f"trunc{i}_v"], rtol=1e-12)
    for key, fn in (("A", positive.A), ("r", positive.r), ("v", positive.v)):
        assert_allclose(fn(g["pos_a"], g["pos_b"]), g[f"pos_{key}"], rtol=1e-12)
    assert isinstance(positive.r(1.0, 0.3), float)
    assert_allclose(positive.tau(2.0, 0.5), positive.r(2.0, 0.5)**2 + positive.v(2.0, 0.5), rtol=1e-14)


def test_size_independent_properties_at_a_small_shape(emulated_device):  # noqa: F811
    """The property checks tests/test_gpu_sizes.py runs on the GPU at N = 4096, here
    at N = 96 through the emulated sweep: the closed forms, tolerances and API calls
    of the checks themselves are pinned by the oracle."""
    from tests import full_size_properties as P
    import torch
    torch.manual_seed(0)
    data = P.make_batch(3, 96, 48, seed=11)
    ref = P.schedules_agree(data, 25)
    assert ref[0].shape == (3, 96) and ref[1].shape == (3,) and ref[2].shape == (25, 3)
    P.oracle_sample(data, ref, b=1, n_iter=25)
    P.instances_are_independent(data, ref, 1, 3, 25)
    P.bayes_optimal_consistency(ref, rtol=2.0, gain=1.0)
    P.linear_gaussian_closed_form(data)


@pytest.mark.parametrize("idx", [0, 1])
def test_jacobi_setup_feeds_the_same_sweep(emulated_device, sw, idx):  # noqa: F811
    """LinearChannel(W, svd_method="jacobi"): the batched block-Jacobi factorisation
    (wide and tall W) gives the reference's spectrum, rank and EP trajectory."""
    from tramp_b200.algos import ExpectationPropagation, TrackErrors
    from tramp_b200.priors import get_prior
    from tramp_b200.likelihoods import get_likelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    W = sw[name + "_W"]
    pk = {k: v for k, v in cfg["prior"].items() if k != "kind"}
    lk = {k: v for k, v in cfg["lik"].items() if k != "kind"}
    lin = LinearChannel(W, svd_method="jacobi")
    model = (get_prior(size=cfg["N"], prior_type=cfg["prior"]["kind"], **pk) @ V("x") @ lin @ V("z")
             @ get_likelihood(y=sw[name + "_y"], likelihood_type=cfg["lik"]["kind"], **lk)).to_model()
    ep = ExpectationPropagation(model)
    track = TrackErrors({"x": sw[name + "_x"]})
    ep.iterate(max_iter=cfg["n_iter"], callback=track, damping=cfg["damping"])
    assert_allclose(lin.s.cpu().numpy()[0], np.linalg.svd(W, compute_uv=False), rtol=1e-11)
    assert lin.rank == np.linalg.matrix_rank(W)
    assert_allclose(np.array([e["mse"] for e in track.errors]), sw[name + "_mse"], rtol=1e-9)
    ref = sw[name + "_rx"]
    assert_allclose(ep.get_variables_data()["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())


def test_smoke_body_and_no_oracle_inside_the_package(emulated_device):  # noqa: F811
    """__graft_entry__.smoke()'s body runs (emulated sweep), and nothing under
    tramp_b200/ imports oracle/: the oracle is the checker, never the product path."""
    import __graft_entry__ as entry
    assert entry._run_smoke(np) < 1e-9
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    for folder, _, files in os.walk(os.path.join(root, "tramp_b200")):
        for name in files:
            if name.endswith(".py"):
                text = open(os.path.join(folder, name)).read()
                assert "import oracle" not in text and "from oracle" not in text, os.path.join(folder, name)


EDGE_OF = {("x", "fwd"): ("e1", "e2"), ("z", "fwd"): ("e3", "e4"), ("z", "bwd"): ("e5", "e6"),
           ("x", "bwd"): ("e7", "e8")}


@pytest.mark.parametrize("seed", range(16))
def test_options_reach_the_right_edges(emulated_device, seed):  # noqa: F811
    """Random models, damping specifications (None / float / per-edge list), initialisers
    (ConstantInit / CustomInit on random edges) and stopping rules through the public API,
    against a direct oracle run given the same choices by edge NAME (SURVEY 3.3: e1 prior->x,
    e3 lin->z, e5 lik->z, e7 lin->x; the variable->factor edges e2/e4/e6/e8 take the
    initial values of their (variable, direction) pair).  What is under test is the mapping
    of (variable id, direction) options into the sweep descriptor."""
    from oracle import tramp_oracle as orc
    from tramp_b200.algos import (ExpectationPropagation, TrackErrors, EarlyStoppingEP, JoinCallback,
                                  ConstantInit, CustomInit)
    from tramp_b200.priors import get_prior
    from tramp_b200.likelihoods import get_likelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    rng = np.random.RandomState(100 + seed)
    N, M = int(rng.randint(20, 60)), int(rng.randint(10, 80))
    pk = ["gauss_bernoulli", "binary", "gaussian"][seed % 3]
    lk = ["gaussian", "sgn", "abs"][(seed // 3) % 3]
    pkw = dict(gauss_bernoulli=dict(rho=0.3), binary=dict(p_pos=0.6), gaussian=dict(mean=0.1, var=0.8))[pk]
    lkw = dict(gaussian=dict(var=0.05), sgn={}, abs={})[lk]
    W = rng.randn(M, N) / np.sqrt(N)
    x = dict(gauss_bernoulli=rng.randn(N) * (rng.rand(N) < 0.3), binary=np.where(rng.rand(N) < 0.6, 1.0, -1.0),
             gaussian=0.1 + np.sqrt(0.8) * rng.randn(N))[pk]
    z = W @ x
    y = dict(gaussian=z + np.sqrt(0.05) * rng.randn(M), sgn=np.where(z >= 0, 1.0, -1.0), abs=np.abs(z))[lk]
    pairs = list(EDGE_OF)
    # damping
    mode = seed % 4
    if mode == 0:
        damping, damp_by_edge = None, None
    elif mode == 1:
        damping, damp_by_edge = 0.3, 0.3
    else:
        chosen = [pairs[k] for k in rng.choice(4, size=rng.randint(1, 4), replace=False)]
        values = [float(rng.choice([0.1, 0.25, 0.5])) for _ in chosen]
        damping = [(vid, direction, d) for (vid, direction), d in zip(chosen, values)]
        damp_by_edge = {EDGE_OF[p][0]: d for p, d in zip(chosen, values)}
    # initial messages
    init_by_edge = {}
    if seed % 3 == 0:
        initializer = None
    elif seed % 3 == 1:
        initializer = ConstantInit(a=0.2, b=0.05)
        for e, n in (("e1", N), ("e2", N), ("e7", N), ("e8", N), ("e3", M), ("e4", M), ("e5", M), ("e6", M)):
            init_by_edge[e] = (0.2, np.full(n, 0.05))
    else:
        a_init, b_init = [], []
        chosen = {}
        for vid, direction in [pairs[k] for k in rng.choice(4, size=2, replace=False)]:
            n = N if vid == "x" else M
            a0, b0 = float(rng.uniform(0.1, 1.0)), 0.1 * rng.randn(n)
            a_init.append((vid, direction, a0))
            b_init.append((vid, direction, b0))
            chosen[vid] = (direction, a0, b0)       # the reference keeps ONE entry per variable id: the last
        for vid, (direction, a0, b0) in chosen.items():
            for e in EDGE_OF[(vid, direction)]:
                init_by_edge[e] = (a0, b0)
        initializer = CustomInit(a_init=a_init, b_init=b_init)
        for e, n in (("e1", N), ("e2", N), ("e7", N), ("e8", N), ("e3", M), ("e4", M), ("e5", M), ("e6", M)):
            init_by_edge.setdefault(e, (0, np.zeros(n)))
    early = seed % 2 == 0
    max_iter = 25
    model = (get_prior(size=N, prior_type=pk, **pkw) @ V("x") @ LinearChannel(W) @ V("z")
             @ get_likelihood(y=y, likelihood_type=lk, **lkw)).to_model()
    ep = ExpectationPropagation(model)
    track = TrackErrors({"x": x})
    callback = JoinCallback([track, EarlyStoppingEP(tol=1e-4)]) if early else track
    with np.errstate(all="ignore"):
        ep.iterate(max_iter=max_iter, callback=callback, initializer=initializer, damping=damping)
        ref = orc.ep_glm(dict(kind=pk, **pkw), W, dict(kind=lk, y=y, **lkw), max_iter, damping=damp_by_edge,
                         init=init_by_edge or None, x_true=x,
                         early_stopping=dict(tol=1e-4) if early else None)
    mse = np.array([e["mse"] for e in track.errors])
    if max(float(np.max(a)) for a, _ in ref["edges"].values()) > 1e4:
        # exact recovery: precisions saturate towards AMAX and the reference's own formulas
        # cancel (DESIGN 6), undamped runs can even oscillate; the first iterations, which
        # already carry the initial messages and the damping, are what can be compared
        assert_allclose(mse[:2], np.array(ref["traj"]["mse_x"])[:2], rtol=1e-7, atol=1e-12)
        return
    assert ep.n_iter == ref["n_iter"]
    got = ep.get_variables_data()
    scale = max(1.0, np.abs(ref["r_x"]).max())
    assert_allclose(got["x"]["r"], ref["r_x"], rtol=1e-9, atol=1e-9 * scale)
    assert_allclose(got["x"]["v"], ref["v_x"], rtol=1e-8, atol=1e-12)
    assert_allclose(got["z"]["v"], ref["v_z"], rtol=1e-8, atol=1e-12)
    assert_allclose(mse, np.array(ref["traj"]["mse_x"])[:len(mse)], rtol=1e-8, atol=1e-14)


def test_reset_precision_bounds_reaches_the_sweep(emulated_device, sw):  # noqa: F811
    """Factor.reset_precision_bounds (reference base.py:241-243): the clip bounds of the
    prior's, the channel's and the likelihood's new precisions travel in the descriptors."""
    from oracle import tramp_oracle as orc
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import SgnLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    rng = np.random.RandomState(5)
    N, M = 40, 90
    W = rng.randn(M, N) / np.sqrt(N)
    x = rng.randn(N) * (rng.rand(N) < 0.3)
    y = np.where(W @ x >= 0, 1.0, -1.0)
    results = {}
    for bounds in (None, (1e-2, 3.0)):
        prior, lik, lin = GaussBernoulliPrior(size=N, rho=0.3), SgnLikelihood(y=y), LinearChannel(W)
        pspec, lspec = dict(kind="gauss_bernoulli", rho=0.3), dict(kind="sgn", y=y)
        op = orc.LinearOp(W)
        if bounds:
            for factor in (prior, lik, lin):
                factor.reset_precision_bounds(*bounds)
            pspec.update(AMIN=bounds[0], AMAX=bounds[1])
            lspec.update(AMIN=bounds[0], AMAX=bounds[1])
            op.AMIN, op.AMAX = bounds
        ep = ExpectationPropagation((prior @ V("x") @ lin @ V("z") @ lik).to_model())
        ep.iterate(max_iter=12, callback=PassCallback(), damping=0.2)
        with np.errstate(all="ignore"):
            ref = orc.ep_glm(pspec, W, lspec, 12, damping=0.2, op=op)
        got = ep.get_variables_data()
        assert_allclose(got["x"]["r"], ref["r_x"], rtol=1e-9, atol=1e-12)
        assert_allclose(got["z"]["v"], ref["v_z"], rtol=1e-9)
        results[bounds] = (got["x"]["r"], max(float(ep._edge(e)[0]) for e in ("e1", "e3", "e5", "e7")))
    assert results[(1e-2, 3.0)][1] <= 3.0 < results[None][1]          # the bounds bind, and change the run
    assert np.abs(results[None][0] - results[(1e-2, 3.0)][0]).max() > 1e-3
