"""GPU parity of the public (tramp-compatible) API against the golden vectors
of the reference and the CPU oracle.  Tolerance: 1e-9 relative on posterior
means / variances and on the MSE trajectory (BASELINE.json north star)."""
import json
import os
import numpy as np
import pytest
from numpy.testing import assert_allclose

from tests.golden import load_sweeps

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module", autouse=True)
def _need_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")


@pytest.fixture(scope="module")
def sw(golden_dir):
    return load_sweeps(golden_dir)


def _configs(sw):
    return json.loads(str(sw["configs"]))


def _build(cfg, sw, name, batch=None):
    from tramp_b200.priors import get_prior
    from tramp_b200.likelihoods import get_likelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    pk = {k: v for k, v in cfg["prior"].items() if k != "kind"}
    lk = {k: v for k, v in cfg["lik"].items() if k != "kind"}
    prior = get_prior(size=cfg["N"], prior_type=cfg["prior"]["kind"], **pk)
    lik = get_likelihood(y=sw[name + "_y"], likelihood_type=cfg["lik"]["kind"], **lk)
    return (prior @ V("x") @ LinearChannel(sw[name + "_W"]) @ V("z") @ lik).to_model()


class _SeqInit:
    """Initializer replaying the eight per-edge initial messages NoisyInit drew
    in the reference run (tests/golden/make_golden.py stores them as e1..e8)."""

    def __init__(self, sw, name):
        self.vals = {k: (float(sw[f"{name}_init_e{k}_a"]), sw[f"{name}_init_e{k}_b"]) for k in range(1, 9)}
        self.calls = 0

    def init(self, key, shape, id, direction):
        # init_message_dag asks a then b, edges in the reference's order (message_dag.edges())
        edge = (1, 2, 8, 3, 7, 4, 6, 5)[(self.calls // 2) % 8]
        self.calls += 1
        return self.vals[edge][0 if key == "a" else 1]


def test_noisy_init_consumes_the_random_stream_like_the_reference(sw):
    """Same seed, same initial messages: NoisyInit is asked for the edges in the order of the
    reference's `message_dag.edges()` (message_passing.py:223-230), so seeding numpy as the golden
    run did reproduces the eight initial messages it recorded -- and hence its whole trajectory."""
    from tramp_b200.algos import ExpectationPropagation, NoisyInit, TrackErrors
    cfg = next(c for c in _configs(sw) if c.get("init") == "noisy")
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, sw, name))
    init = NoisyInit(a_mean=0.5, a_var=0, b_mean=0, b_var=0.25)
    np.random.seed(cfg["seed"] + 1000)
    ep.init_message_dag(init)
    for k in range(1, 9):
        a, b = ep._edge(f"e{k}") if k in (1, 2, 3, 4, 5, 7) else (None, None)
        if a is not None and k in (1, 3, 5, 7):
            assert_allclose(a, float(sw[f"{name}_init_e{k}_a"]), rtol=0, atol=0)
            assert np.array_equal(b, sw[f"{name}_init_e{k}_b"])
    track = TrackErrors({"x": sw[name + "_x"]})
    np.random.seed(cfg["seed"] + 1000)
    ep.iterate(max_iter=cfg["n_iter"], callback=track, initializer=init, damping=cfg["damping"])
    ref = sw[name + "_mse"]
    tau_x = np.mean(sw[name + "_x"]**2)
    mse = np.array([e["mse"] for e in track.errors])
    assert np.all(np.abs(mse - ref) <= 1e-9 * ref + 2e-9 * np.sqrt(ref * tau_x))


@pytest.mark.parametrize("impl,schedule", [(1, "general"), (2, "general"), (2, "auto")])
@pytest.mark.parametrize("idx", range(9))
def test_sweep_matches_reference(sw, idx, impl, schedule):
    """schedule "general" = 4 operator passes per iteration; "auto" picks the exact
    3-pass (damped) / 2-pass (undamped) schedules when the likelihood is Gaussian."""
    from tramp_b200.algos import ExpectationPropagation, TrackErrors, TrackEvolution, JoinCallback
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    model = _build(cfg, sw, name)
    ep = ExpectationPropagation(model)
    ep.gemv_impl = impl
    ep.schedule = schedule
    track = TrackErrors({"x": sw[name + "_x"]})
    evo = TrackEvolution()
    init = _SeqInit(sw, name) if cfg.get("init") == "noisy" else None
    ep.iterate(max_iter=cfg["n_iter"], callback=JoinCallback([track, evo]), initializer=init,
               damping=cfg["damping"])
    assert ep.n_iter == cfg["n_iter"]
    if schedule == "general":
        assert ep.last_schedule == 0
    elif cfg["lik"]["kind"] == "gaussian" and cfg.get("init") != "noisy":
        assert ep.last_schedule == (1 if cfg["damping"] else 2)
    mse = np.array([e["mse"] for e in track.errors])
    df = evo.get_dataframe()
    x, W = sw[name + "_x"], sw[name + "_W"]
    tau_x, tau_z = np.mean(x**2), np.mean((W @ x)**2)
    # Tolerance: 1e-9 relative.  At exact recovery (binary / noiseless configs,
    # a -> 1e6..AMAX) the reference's own formulas cancel (1 - tanh^2, 1/v - a),
    # so a quantity q is also accepted within 1e-9 of its natural scale: the
    # signal's second moment for variances, sqrt(mse * tau) for the MSE (i.e. r
    # within 1e-9 of the signal scale), max|r| for means.  See DESIGN.md "Parity".
    ref = sw[name + "_mse"]
    assert np.all(np.abs(mse - ref) <= 1e-9 * ref + 2e-9 * np.sqrt(ref * tau_x))
    assert_allclose(df[df.id == "x"].v.values, sw[name + "_vx"], rtol=1e-9, atol=1e-9 * tau_x)
    assert_allclose(df[df.id == "z"].v.values, sw[name + "_vz"], rtol=1e-9, atol=1e-9 * tau_z)
    d = ep.get_variables_data()
    for vid, key in (("x", "_rx"), ("z", "_rz")):
        ref = sw[name + key]
        assert_allclose(d[vid]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    assert_allclose(d["x"]["v"], sw[name + "_vx_final"], rtol=1e-9, atol=1e-9 * tau_x)
    assert_allclose(d["z"]["v"], sw[name + "_vz_final"], rtol=1e-9, atol=1e-9 * tau_z)
    # individual messages are compared where they are well conditioned; in the
    # saturated regime (some a > 1e4) only the posteriors above are meaningful
    saturated = max(float(sw[f"{name}_e{k}_a"]) for k in range(1, 9)) > 1e4
    for k in range(1, 9):
        a, b = ep._edge(f"e{k}")
        ref_b = sw[f"{name}_e{k}_b"]
        if saturated:
            assert np.isfinite(a) and np.all(np.isfinite(b))
            continue
        assert_allclose(a, sw[f"{name}_e{k}_a"], rtol=1e-9)
        assert_allclose(b, ref_b, rtol=1e-9, atol=1e-9 * np.abs(ref_b).max())


@pytest.mark.parametrize("idx", range(9))
def test_log_evidence_matches_reference(sw, idx):
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, sw, name))
    init = _SeqInit(sw, name) if cfg.get("init") == "noisy" else None
    ep.iterate(max_iter=cfg["n_iter"], callback=PassCallback(), initializer=init, damping=cfg["damping"])
    with np.errstate(all="ignore"):
        logZ = ep.log_evidence()
    saturated = max(float(sw[f"{name}_e{k}_a"]) for k in range(1, 9)) > 1e4
    if saturated:
        # a -> 1e6..AMAX: log Z is a difference of ~1e8..1e13 terms built from
        # messages that are themselves ill conditioned (see test_sweep_matches_reference)
        assert np.isfinite(logZ)
        assert_allclose(logZ, sw[name + "_logZ"], rtol=1e-2)
        return
    # A_model = sum(nodes) - sum(edges): tolerance relative to the size of the terms
    scale = sum(abs(v) for v in ep.A_nodes.values()) + sum(abs(v) for v in ep.A_edges.values())
    assert abs(logZ - sw[name + "_logZ"]) <= 1e-9 * scale
    assert_allclose(ep.A_nodes[ep.prior.id], sw[name + "_A_" + type(ep.prior).__name__], rtol=1e-9)
    assert_allclose(ep.A_nodes[ep.lik.id], sw[name + "_A_" + type(ep.lik).__name__], rtol=1e-9)
    assert_allclose(ep.A_nodes[ep.linear.id], sw[name + "_A_LinearChannel"], rtol=1e-9)
    assert_allclose(ep.A_nodes["x"], sw[name + "_A_x"], rtol=1e-9)
    assert_allclose(ep.A_nodes["z"], sw[name + "_A_z"], rtol=1e-9)


@pytest.mark.parametrize("idx", range(3))
def test_default_early_stopping(sw, idx):
    """iterate() with the default EarlyStoppingEP stops at the reference's iteration."""
    from tramp_b200.algos import ExpectationPropagation
    cfg = _configs(sw)[idx]
    name = cfg["name"] + "_early"
    ep = ExpectationPropagation(_build(cfg, sw, name))
    ep.iterate(max_iter=200, damping=cfg["damping"])
    assert ep.n_iter == int(sw[name + "_n_iter"])
    d = ep.get_variables_data()
    ref = sw[name + "_rx"]
    assert_allclose(d["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    assert_allclose(d["x"]["v"], sw[name + "_vx_final"], rtol=1e-9)


def test_early_stopping_divergence_restores_previous_iteration(sw):
    """EarlyStoppingEP's max_increase branch (callbacks.py:275-283) on the device:
    the instance is frozen AND rolled back to the end of the previous iteration."""
    from tramp_b200.algos import ExpectationPropagation, TrackEstimate, JoinCallback, EarlyStoppingEP
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    name = "cs_diverges_early"

    def build():
        return (GaussBernoulliPrior(size=120, rho=0.1) @ V("x") @ LinearChannel(sw[name + "_W"]) @ V("z")
                @ GaussianLikelihood(y=sw[name + "_y"], var=1e-2)).to_model()
    for callback in (None, JoinCallback([TrackEstimate(ids=["x"]), EarlyStoppingEP()])):   # device / host path
        ep = ExpectationPropagation(build())
        ep.iterate(max_iter=200, callback=callback)
        assert ep.n_iter == int(sw[name + "_n_iter"]) == 7
        d = ep.get_variables_data()
        assert_allclose(d["x"]["r"], sw[name + "_rx"], rtol=1e-9, atol=1e-12)
        assert_allclose(d["z"]["r"], sw[name + "_rz"], rtol=1e-9, atol=1e-12)
        assert_allclose(d["x"]["v"], sw[name + "_vx_final"], rtol=1e-9)
        for k in range(1, 9):
            a, b = ep._edge(f"e{k}")
            assert_allclose(a, sw[f"{name}_e{k}_a"], rtol=1e-9)
            assert_allclose(b, sw[f"{name}_e{k}_b"], rtol=1e-9, atol=1e-12)


def test_synchronous_callback_path_equals_device_path(sw):
    """An arbitrary callback (TrackEstimate needs r every iteration) forces the
    per-iteration path; it must give the same trajectory as the device path."""
    from tramp_b200.algos import (ExpectationPropagation, TrackErrors, TrackEstimate,
                                  JoinCallback, EarlyStoppingEP)
    cfg = _configs(sw)[1]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, sw, name))
    est = TrackEstimate(ids=["x"])
    track = TrackErrors({"x": sw[name + "_x"]})
    ep.iterate(max_iter=cfg["n_iter"], callback=JoinCallback([est, track]), damping=cfg["damping"])
    mse = np.array([e["mse"] for e in track.errors])
    assert_allclose(mse, sw[name + "_mse"], rtol=1e-9)
    assert len(est.records) == cfg["n_iter"]
    assert_allclose(est.records[-1]["r"], sw[name + "_rx"], rtol=1e-9, atol=1e-12)
    # host-side EarlyStoppingEP (inside a join with a non-replayable callback)
    name_e = cfg["name"] + "_early"
    ep = ExpectationPropagation(_build(cfg, sw, name_e))
    ep.iterate(max_iter=200, callback=JoinCallback([TrackEstimate(ids=["x"]), EarlyStoppingEP()]),
               damping=cfg["damping"])
    assert ep.n_iter == int(sw[name_e + "_n_iter"])


def test_warm_start_continues(sw):
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    cfg = _configs(sw)[0]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, sw, name))
    ep.iterate(max_iter=15, callback=PassCallback())
    ep.iterate(max_iter=cfg["n_iter"] - 15, callback=PassCallback(), warm_start=True)
    assert ep.n_iter == cfg["n_iter"]
    ref = sw[name + "_rx"]
    assert_allclose(ep.get_variables_data()["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    ep2 = ExpectationPropagation(_build(cfg, sw, name))
    with pytest.raises(ValueError):
        ep2.iterate(max_iter=1, warm_start=True)


def test_errors_mirror_reference(sw):
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.channels import LinearChannel, GaussianChannel
    from tramp_b200.variables import SISOVariable as V, SILeafVariable as O
    cfg = _configs(sw)[0]
    ep = ExpectationPropagation(_build(cfg, sw, cfg["name"]))
    with pytest.raises(ValueError):
        ep.iterate(max_iter=1, callback=PassCallback(), damping=1)      # int, not float
    from tramp_b200.algos import MessagePassing
    with pytest.raises(ValueError):
        MessagePassing("not a model", message_keys=["a", "b"])
    # un-observed generative model is not the EP chain
    gen = (GaussBernoulliPrior(size=8) @ V("x") @ LinearChannel(np.eye(8)) @ V("z")
           @ GaussianChannel(var=1.) @ O("y")).to_model()
    with pytest.raises(NotImplementedError):
        ExpectationPropagation(gen)
    # NaN in a message surfaces as ValueError (message_passing.py:187-209)
    name = cfg["name"]
    y_bad = sw[name + "_y"].copy()
    y_bad[3] = np.nan
    from tramp_b200.likelihoods import GaussianLikelihood
    m = (GaussBernoulliPrior(size=cfg["N"], rho=0.1) @ V("x") @ LinearChannel(sw[name + "_W"]) @ V("z")
         @ GaussianLikelihood(y=y_bad, var=1e-2)).to_model()
    with pytest.raises(ValueError, match="nan"):
        ExpectationPropagation(m).iterate(max_iter=3, callback=PassCallback())


@pytest.mark.parametrize("kinds", [("gauss_bernoulli", "gaussian"), ("gaussian", "sgn"),
                                   ("binary", "abs")])
def test_batched_instances_match_oracle(kinds):
    """B independent instances in one launch == B oracle runs (north-star item 4),
    incl. a batch that shares one W (config-4 style)."""
    from oracle import tramp_oracle as orc
    from tramp_b200.priors import get_prior
    from tramp_b200.likelihoods import get_likelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import ExpectationPropagation, TrackErrors
    pk, lk = kinds
    rng = np.random.RandomState(5)
    B, N, M, n_iter, damping = 5, 96, 144 if lk != "gaussian" else 48, 25, 0.3
    pkw = dict(gauss_bernoulli=dict(rho=0.2), gaussian={}, binary=dict(p_pos=0.6))[pk]
    lkw = dict(gaussian=dict(var=0.02), sgn={}, abs={})[lk]
    for shared in (False, "gemm", "cublas"):
        W = rng.randn(*(() if shared else (B,)), M, N) / np.sqrt(N)
        if pk == "gauss_bernoulli":
            x = rng.randn(B, N) * (rng.rand(B, N) < 0.2)
        elif pk == "binary":
            x = np.where(rng.rand(B, N) < 0.6, 1.0, -1.0)
        else:
            x = rng.randn(B, N)
        Wb = np.broadcast_to(W, (B, M, N))
        z = np.einsum("bmn,bn->bm", Wb, x)
        y = dict(gaussian=z + np.sqrt(0.02) * rng.randn(B, M), sgn=np.where(z >= 0, 1., -1.),
                 abs=np.abs(z))[lk]
        model = (get_prior(size=N, prior_type=pk, batch=B, **pkw) @ V("x") @ LinearChannel(W) @ V("z")
                 @ get_likelihood(y=y, likelihood_type=lk, **lkw)).to_model()
        ep = ExpectationPropagation(model)
        if shared:
            # shared W: the four passes become FP64 GEMMs -- "gemm" = the DMMA kernels
            # of trb_gemm.cu inside trb_sweep_run, "cublas" = the library baseline
            ep.linear_backend = shared
        track = TrackErrors({"x": x}, metrics=["mse", "sign_mse"])
        ep.iterate(max_iter=n_iter, callback=track, damping=damping)
        assert ep.backend == (shared or "gemv")
        got = ep.get_variables_data()
        assert got["x"]["r"].shape == (B, N) and got["x"]["v"].shape == (B,)
        for b in range(B):
            with np.errstate(all="ignore"):
                ref = orc.ep_glm(dict(kind=pk, **pkw), Wb[b], dict(kind=lk, y=y[b], **lkw), n_iter,
                                 damping=damping, x_true=x[b])
            for vid, r in (("x", ref["r_x"]), ("z", ref["r_z"])):
                assert_allclose(got[vid]["r"][b], r, rtol=1e-9, atol=1e-9 * np.abs(r).max())
            assert_allclose(got["x"]["v"][b], ref["v_x"], rtol=1e-9)
            assert_allclose(got["z"]["v"][b], ref["v_z"], rtol=1e-9)
            mse = np.array([e["mse"][b] for e in track.errors])
            ref_mse = np.array(ref["traj"]["mse_x"])
            # 1e-9 relative, or r within 1e-9 of the signal scale at exact recovery
            assert np.all(np.abs(mse - ref_mse) <= 1e-9 * ref_mse + 2e-9 * np.sqrt(ref_mse * np.mean(x[b]**2)))
            smse = np.array([e["sign_mse"][b] for e in track.errors])
            assert np.all(smse <= mse * (1 + 1e-12))


def test_batched_early_stopping_per_instance():
    """Each instance of a batch stops at the iteration its own oracle run stops."""
    from oracle import tramp_oracle as orc
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import ExpectationPropagation
    rng = np.random.RandomState(9)
    B, N, M = 4, 120, 60
    W = rng.randn(B, M, N) / np.sqrt(N)
    x = rng.randn(B, N) * (rng.rand(B, N) < 0.1)
    y = np.einsum("bmn,bn->bm", W, x) + 0.1 * rng.randn(B, M)
    model = (GaussBernoulliPrior(size=N, rho=0.1, batch=B) @ V("x") @ LinearChannel(W) @ V("z")
             @ GaussianLikelihood(y=y, var=1e-2)).to_model()
    ep = ExpectationPropagation(model)
    ep.iterate(max_iter=200)
    got = ep.get_variables_data()
    for b in range(B):
        ref = orc.ep_glm(dict(kind="gauss_bernoulli", rho=0.1), W[b],
                         dict(kind="gaussian", var=1e-2, y=y[b]), 200,
                         early_stopping=dict(tol=1e-6))
        assert ep.n_iter_per_instance[b] == ref["n_iter"]
        assert_allclose(got["x"]["r"][b], ref["r_x"], rtol=1e-9, atol=1e-12)
    assert ep.n_iter == ep.n_iter_per_instance.max()


def test_factor_api_mirrors_reference_unit_tests():
    """tramp/tests/test_priors.py:27-52 and test_likelihoods.py:52-86: vectorised
    compute_*_posterior / compute_log_partition equal the scalar_* versions, with
    isotropic=False and ax in linspace(1, 2), bx in linspace(-2, 2)."""
    from tramp_b200.priors import GaussianPrior, GaussBernoulliPrior, BinaryPrior
    from tramp_b200.likelihoods import GaussianLikelihood, AbsLikelihood, SgnLikelihood
    ax = np.linspace(1, 2, 100)
    bx = np.linspace(-2, 2, 100)
    for prior in (GaussianPrior(size=100, isotropic=False), GaussBernoulliPrior(size=100, isotropic=False),
                  BinaryPrior(size=100, isotropic=False)):
        rx, vx = prior.compute_forward_posterior(ax, bx)
        assert rx.shape == bx.shape and vx.shape == bx.shape
        rx_ = np.array([prior.scalar_forward_mean(a, b) for a, b in zip(ax, bx)])
        vx_ = np.array([prior.scalar_forward_variance(a, b) for a, b in zip(ax, bx)])
        assert_allclose(rx, rx_)
        assert_allclose(vx, vx_)
        A = prior.compute_log_partition(ax, bx)
        A_ = np.mean([prior.scalar_log_partition(a, b) for a, b in zip(ax, bx)])
        assert_allclose(A, A_, rtol=1e-13)
    z = np.linspace(-3, 3, 100)
    for lik in (GaussianLikelihood(y=z, isotropic=False), AbsLikelihood(y=np.abs(z), isotropic=False),
                SgnLikelihood(y=np.sign(z), isotropic=False)):
        rz, vz = lik.compute_backward_posterior(ax, bx, lik.y)
        assert rz.shape == bx.shape and vz.shape == bx.shape
        rz_ = np.array([lik.scalar_backward_mean(a, b, y) for a, b, y in zip(ax, bx, lik.y)])
        vz_ = np.array([lik.scalar_backward_variance(a, b, y) for a, b, y in zip(ax, bx, lik.y)])
        assert_allclose(rz, rz_)
        assert_allclose(vz, vz_)
        A = lik.compute_log_partition(ax, bx, lik.y)
        A_ = np.mean([lik.scalar_log_partition(a, b, y) for a, b, y in zip(ax, bx, lik.y)])
        assert_allclose(A, A_, rtol=1e-13)


def test_belief_gradients():
    """tramp/tests/test_beliefs.py:11-23 (checks/check_gradients.py:44,70-90):
    r = dA/db and v = d2A/db2 by central finite differences, eps = 1e-3, atol 1e-3."""
    from tramp_b200.beliefs import binary, normal, sparse, positive, truncated
    eps = 1e-3
    b = np.linspace(-6, 6, 100)
    cases = [(binary, {}), (normal, {"a": 1}), (sparse, {"a": 1, "eta": 1}), (positive, {"a": 1}),
             (truncated, {"a": 1, "xmin": -1, "xmax": +1})]
    for belief, kw in cases:
        def A(bb):
            return belief.A(b=bb, **kw)
        A1 = (A(b + eps) - A(b - eps)) / (2 * eps)
        A2 = (A(b + eps) - 2 * A(b) + A(b - eps)) / eps**2
        assert_allclose(belief.r(b=b, **kw), A1, rtol=0, atol=eps)
        assert_allclose(belief.v(b=b, **kw), A2, rtol=0, atol=eps)


def test_beliefs_against_reference(golden_dir):
    """Every function of tramp/beliefs/{sparse,binary,positive,truncated}.py against the reference
    (tests/golden/beliefs.npz), including the weight `sparse.p` down to 1e-18 (reference
    beliefs/sparse.py:9-12: expit(normal.A - eta)), 1e-11 relative."""
    from tramp_b200.beliefs import binary, sparse, positive, truncated
    g = np.load(os.path.join(golden_dir, "beliefs.npz"))
    a, b = g["bel_a"], g["bel_b"]
    tiny = 1e-300
    for k, eta in enumerate(g["sparse_eta"]):
        for name in ("A", "p", "r", "v", "tau"):
            ref = g[f"sparse{k}_{name}"]
            got = getattr(sparse, name)(a, b, float(eta))
            # v = s / a + s (1 - s) (b / a)^2 and tau are sums of positive terms: plain relative
            assert_allclose(got, ref, rtol=1e-11, atol=tiny, err_msg=f"sparse.{name} eta={eta}")
    assert g["sparse7_p"].min() < 1e-17                      # the regime 1 - exp(eta - A) cannot reach
    bb = g["binary_b"]
    assert_allclose(binary.A(bb), g["binary_A"], rtol=1e-13)
    assert_allclose(binary.r(bb), g["binary_r"], rtol=1e-13)
    # 1 - tanh^2 cancels for |b| >> 1: the reference's own rounding is eps absolute
    assert_allclose(binary.v(bb), g["binary_v"], rtol=1e-11, atol=4 * np.finfo(float).eps)
    for name in ("A", "r", "v", "tau", "p"):
        ref = g[f"positive_{name}"]
        got = getattr(positive, name)(a, b)
        assert_allclose(got, ref, rtol=1e-10, atol=1e-13 * np.abs(ref).max(), err_msg=f"positive.{name}")
    bt = g["trunc_b"]
    for i, (a_t, lo, hi) in enumerate(g["trunc_cases"]):
        for name in ("tau", "p"):
            ref = g[f"trunc{i}_{name}"]
            ok = np.isfinite(ref)
            got = getattr(truncated, name)(a_t, bt, lo, hi)
            assert_allclose(got[ok], ref[ok], rtol=1e-9, atol=1e-13, err_msg=f"truncated.{name} case {i}")


def test_linear_channel_reference_signature_corners():
    """The corners of the reference constructor / factor API (channels/linear/linear_channel.py):
    `precompute_svd=False` (:43-45, :79-82: dense solve per call -- same numbers), `bz` of shape
    [Nz, k] with one scalar precision (:75-76), and the free energies of a batched channel (:134-143)."""
    from tramp_b200.channels import LinearChannel
    rng = np.random.RandomState(9)
    Nx, Nz, k = 30, 20, 3
    W = rng.randn(Nx, Nz) / np.sqrt(Nz)
    az, ax = 0.7, 2.5
    bz, bx = rng.randn(Nz), rng.randn(Nx)
    lazy, eager = LinearChannel(W, precompute_svd=False), LinearChannel(W)
    assert lazy.precompute_svd is False and "precompute_svd=False" in repr(lazy)
    C = W.T @ W
    rz_ref = np.linalg.solve(az * np.identity(Nz) + ax * C, bz + W.T @ bx)            # reference :79-82
    for ch in (lazy, eager):
        assert_allclose(ch.compute_backward_mean(az, bz, ax, bx), rz_ref, rtol=1e-11, atol=1e-13)
        assert_allclose(ch.compute_forward_mean(az, bz, ax, bx), W @ rz_ref, rtol=1e-11, atol=1e-13)
    assert_allclose(np.sort(lazy.spectrum), np.linalg.eigvalsh(C), rtol=1e-11, atol=1e-14)
    assert lazy.compute_backward_variance(az, ax) == eager.compute_backward_variance(az, ax)
    # a block of k columns, one scalar az / ax (reference :75-76)
    Bz, Bx = rng.randn(Nz, k), rng.randn(Nx, k)
    Rz = eager.compute_backward_mean(az, Bz, ax, Bx)
    assert Rz.shape == (Nz, k)
    assert_allclose(Rz, np.linalg.solve(az * np.identity(Nz) + ax * C, Bz + W.T @ Bx), rtol=1e-11, atol=1e-13)
    Rx, vx = eager.compute_forward_posterior(az, Bz, ax, Bx)
    assert Rx.shape == (Nx, k) and np.ndim(vx) == 0
    assert_allclose(Rx, W @ Rz, rtol=1e-11, atol=1e-13)
    assert vx == eager.compute_forward_variance(az, ax)
    with pytest.raises(ValueError, match="one scalar"):
        eager.compute_backward_mean(np.array([0.5, 0.6, 0.7]), Bz, ax, Bx)
    # batched channel: one mutual information / free energy per instance
    Wb = rng.randn(3, Nx, Nz) / np.sqrt(Nz)
    batch = LinearChannel(Wb)
    I = batch.compute_mutual_information(az, ax, tau_z=1.3)
    A = batch.compute_free_energy(az, ax, tau_z=1.3)
    assert I.shape == (3,) and A.shape == (3,)
    for b in range(3):
        one = LinearChannel(Wb[b])
        spectrum = np.linalg.eigvalsh(Wb[b].T @ Wb[b])
        assert_allclose(I[b], np.mean(0.5 * np.log((az + ax * spectrum) * 1.3)), rtol=1e-11)    # reference :134-137
        assert_allclose(I[b], one.compute_mutual_information(az, ax, 1.3), rtol=1e-13)
        assert_allclose(A[b], one.compute_free_energy(az, ax, 1.3), rtol=1e-13)


def test_linear_channel_factor_api(golden_dir):
    """LinearChannel.compute_*_posterior / log_partition against the reference."""
    from tramp_b200.channels import LinearChannel
    lin = np.load(os.path.join(golden_dir, "linear.npz"))
    for i in range(int(lin["lin_nW"])):
        ch = LinearChannel(lin[f"lin{i}_W"])
        bz, bx = lin[f"lin{i}_bz"], lin[f"lin{i}_bx"]
        assert ch._setup() is None and ch.rank == int(lin[f"lin{i}_rank"])
        for j, (az, ax) in enumerate(lin["lin_ab"]):
            if az == 0:
                continue
            rz, vz = ch.compute_backward_posterior(az, bz, ax, bx)
            rx, vx = ch.compute_forward_posterior(az, bz, ax, bx)
            # reference rx = W @ rz loses eps*|rz| absolutely when az << ax (see
            # test_gpu_primitives.test_linear_channel_primitives)
            noise = 64 * np.finfo(float).eps * np.abs(lin[f"lin{i}_{j}_rz"]).max()
            for got, key in ((rz, "rz"), (rx, "rx")):
                ref = lin[f"lin{i}_{j}_{key}"]
                assert_allclose(got, ref, rtol=1e-9, atol=max(noise, 1e-12 * max(1.0, np.abs(ref).max())))
            assert_allclose(vz, lin[f"lin{i}_{j}_vz"], rtol=1e-12,
                            atol=16 * np.finfo(float).eps / max(az, 1e-11))   # 1 - n_eff cancels
            assert_allclose(vx, lin[f"lin{i}_{j}_vx"], rtol=1e-12)
            assert_allclose(ch.compute_n_eff(az, ax), lin[f"lin{i}_{j}_neff"], rtol=1e-10)
            with np.errstate(all="ignore"):
                A = ch.compute_log_partition(az, bz, ax, bx)
            assert_allclose(A, lin[f"lin{i}_{j}_A"], rtol=1e-9)


@pytest.mark.parametrize("idx", [0, 2, 5])
def test_gram_factorisation_matches_reference(sw, idx):
    """svd_method="auto" factorises a well-conditioned W through the eigen-
    decomposition of its smaller Gram matrix (cheaper set-up); the sweep still
    matches the reference to 1e-9."""
    from tramp_b200.algos import ExpectationPropagation, TrackErrors
    from tramp_b200.priors import get_prior
    from tramp_b200.likelihoods import get_likelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.channels.linear_channel import thin_svd_device
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200 import ops
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    W = sw[name + "_W"]
    pk = {k: v for k, v in cfg["prior"].items() if k != "kind"}
    lk = {k: v for k, v in cfg["lik"].items() if k != "kind"}
    lin = LinearChannel(W, svd_method="auto")
    model = (get_prior(size=cfg["N"], prior_type=cfg["prior"]["kind"], **pk) @ V("x") @ lin @ V("z")
             @ get_likelihood(y=sw[name + "_y"], likelihood_type=cfg["lik"]["kind"], **lk)).to_model()
    ep = ExpectationPropagation(model)
    track = TrackErrors({"x": sw[name + "_x"]})
    ep.iterate(max_iter=cfg["n_iter"], callback=track, damping=cfg["damping"])
    s_ref = np.linalg.svd(W, compute_uv=False)
    assert_allclose(lin.s.cpu().numpy()[0], s_ref, rtol=1e-12)
    assert lin.rank == np.linalg.matrix_rank(W)
    mse = np.array([e["mse"] for e in track.errors])
    ref = sw[name + "_mse"]
    tau_x = np.mean(sw[name + "_x"]**2)
    assert np.all(np.abs(mse - ref) <= 1e-9 * ref + 2e-9 * np.sqrt(ref * tau_x))
    ref = sw[name + "_rx"]
    assert_allclose(ep.get_variables_data()["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    # an ill-conditioned matrix falls back to the SVD
    Wd = ops.to_dev(W.copy())[None]
    Wd[0, -1] = Wd[0, 0] * (1 + 1e-9)
    s_auto = thin_svd_device(Wd, "auto")[1]
    s_svd = thin_svd_device(Wd, "svd")[1]
    assert_allclose(s_auto.cpu().numpy(), s_svd.cpu().numpy(), rtol=1e-12, atol=1e-18)


def test_scenario_and_glm_generative():
    """BayesOptimalScenario.setup/run_ep/ep_convergence on glm_generative
    (reference experiments/teacher_student_scenario.py:45-115)."""
    from tramp_b200.models import glm_generative
    from tramp_b200.experiments import BayesOptimalScenario
    np.random.seed(12)
    model = glm_generative(N=200, alpha=0.6, ensemble_type="gaussian", prior_type="gauss_bernoulli",
                           output_type="gaussian", prior_rho=0.1, output_var=1e-2)
    scenario = BayesOptimalScenario(model, x_ids=["x"])
    scenario.setup(seed=42)
    x_data = scenario.run_ep(max_iter=200, damping=0.1)
    mse = np.mean((x_data["x"]["r"] - scenario.x_true["x"])**2)
    assert x_data["n_iter"] < 200
    assert mse < 0.02 and abs(mse - x_data["x"]["v"]) < 0.01   # EP's v tracks the empirical mse
    df = scenario.ep_convergence(metrics=["mse"], max_iter=30, damping=0.1)
    assert list(df.columns) == ["id", "iter", "mse", "v"] and len(df) == 30
    assert_allclose(scenario.compute_score(scenario.x_pred)["x"]["mse"], df.mse.values[-1], rtol=1e-9)


# ---------------------------------------------------------------------------
# host-driven factor-by-factor schedule: damping="adaptive", update_dA, TrackObjective
# ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ad(golden_dir):
    return np.load(os.path.join(golden_dir, "adaptive.npz"))


@pytest.mark.parametrize("idx", range(4))
def test_adaptive_damping_and_dA_match_reference(ad, idx):
    """reference message_passing.py:129-185 run through the unmodified reference
    (tests/golden/make_golden.py section D): trajectories, per-iteration A_model
    (update_objective), final messages with their dA / beta / n_iter."""
    from tramp_b200.algos import ExpectationPropagation, TrackObjective, TrackMessages, JoinCallback
    cfg = json.loads(str(ad["configs"]))[idx]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, ad, name))
    x = ad[name + "_x"]
    rows = []

    def record(algo, i, max_iter):
        d = algo.get_variables_data()
        rows.append((np.mean((d["x"]["r"] - x)**2), d["x"]["v"], d["z"]["v"]))

    obj, msgs = TrackObjective(), TrackMessages(keys=["a", "n_iter", "direction", "dA", "beta"])
    ep.iterate(max_iter=cfg["n_iter"], callback=JoinCallback([record, obj, msgs]),
               damping=cfg["damping"], update_dA=cfg["update_dA"])
    assert ep.n_iter == cfg["n_iter"]
    mse, vx, vz = (np.array(c) for c in zip(*rows))
    assert_allclose(mse, ad[name + "_mse"], rtol=1e-9)
    assert_allclose(vx, ad[name + "_vx"], rtol=1e-9)
    assert_allclose(vz, ad[name + "_vz"], rtol=1e-9)
    edge_df, node_df, model_df = obj.get_dataframe()
    A_ref = ad[name + "_A_model"]
    # A_model = sum(nodes) - sum(edges) of terms ~1e2..1e3: tolerance relative to their size
    assert_allclose(model_df.A.values, A_ref, rtol=1e-9, atol=1e-9 * 1e3)
    assert len(node_df) == 5 * cfg["n_iter"] and len(edge_df) == 8 * cfg["n_iter"]
    d = ep.get_variables_data()
    for vid, key in (("x", "_rx"), ("z", "_rz")):
        ref = ad[name + key]
        assert_allclose(d[vid]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    last = {}
    for rec in msgs.get_dataframe().to_dict("records")[-8:]:
        last[(rec["x_id"], rec["f_id"], rec["direction"])] = rec
    for k in range(1, 9):
        a, b = ep._edge(f"e{k}")
        assert_allclose(a, ad[f"{name}_e{k}_a"], rtol=1e-9)
        ref_b = ad[f"{name}_e{k}_b"]
        assert_allclose(b, ref_b, rtol=1e-9, atol=1e-9 * max(np.abs(ref_b).max(), 1e-300))
        data = ep._host.edges[f"e{k}"]
        assert data["n_iter"] == int(ad[f"{name}_e{k}_n_iter"])
        if cfg["damping"] == "adaptive":
            assert data["beta"] == float(ad[f"{name}_e{k}_beta"])
        ref_dA = float(ad[f"{name}_e{k}_dA"])
        # dA is a difference of objectives of size ~|A_model|
        assert abs(data["dA"] - ref_dA) <= 1e-9 * max(1.0, np.abs(A_ref).max())
    assert len(last) == 8


def test_host_path_then_device_warm_start(ad):
    """update_dA (host path) for a few iterations, then a plain warm-started
    device sweep continues from the same messages: equals one uninterrupted run."""
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    cfg = json.loads(str(ad["configs"]))[2]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, ad, name))
    ep.iterate(max_iter=3, callback=PassCallback(), damping=0.2, update_dA=True)
    ep.iterate(max_iter=5, callback=PassCallback(), damping=0.2, warm_start=True)
    assert ep.n_iter == 8
    d = ep.get_variables_data()
    ref = ad[name + "_rx"]
    assert_allclose(d["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
    assert_allclose(d["x"]["v"], ad[name + "_vx"][-1], rtol=1e-9)


@pytest.mark.parametrize("options", [dict(damping="adaptive"), dict(damping=0.2, update_dA=True)])
def test_adaptive_damping_batched_equals_per_instance(options):
    """damping="adaptive" / update_dA on a BATCH (reference message_passing.py:129-185 has no batches):
    every instance takes its own step-halving decisions, so the batched run reproduces the
    per-instance runs -- posteriors, messages, and the accepted step size beta of every edge."""
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import SgnLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    rng = np.random.RandomState(5)
    B, N, M, n_iter = 3, 40, 60, 6
    W = rng.randn(B, M, N) / np.sqrt(N)
    x = rng.randn(B, N) * (rng.rand(B, N) < 0.3)
    y = np.sign(np.einsum("bmn,bn->bm", W, x))

    def run(Wb, yb, batch):
        model = (GaussBernoulliPrior(size=N, rho=0.3, batch=batch) @ V("x") @ LinearChannel(Wb) @ V("z")
                 @ SgnLikelihood(y=yb)).to_model()
        ep = ExpectationPropagation(model)
        ep.iterate(max_iter=n_iter, callback=PassCallback(), **options)
        return ep
    whole = run(W, y, B)
    assert whole.n_iter == n_iter and whole.n_iter_per_instance.tolist() == [n_iter] * B
    d_all = whole.get_variables_data()
    betas = []
    for b in range(B):
        one = run(W[b], y[b], None)
        d = one.get_variables_data()
        for vid in ("x", "z"):
            assert_allclose(d_all[vid]["r"][b], d[vid]["r"], rtol=1e-10, atol=1e-12)
            assert_allclose(d_all[vid]["v"][b], d[vid]["v"], rtol=1e-10)
        for k in range(1, 9):
            e_all, e_one = whole._host.edges[f"e{k}"], one._host.edges[f"e{k}"]
            assert_allclose(e_all["a"][b], e_one["a"], rtol=1e-10)
            assert_allclose(e_all["b"][b], e_one["b"], rtol=1e-10, atol=1e-12)
            assert_allclose(np.asarray(e_all["dA"])[b] if np.ndim(e_all["dA"]) else e_all["dA"], e_one["dA"],
                            rtol=1e-7, atol=1e-9)
            if options["damping"] == "adaptive":
                assert e_all["beta"][b] == e_one["beta"]
                betas.append(e_one["beta"])
    if options["damping"] == "adaptive":
        assert min(betas) < 1.0 <= max(betas)       # the instances did take different step sizes


@pytest.mark.parametrize("idx", [0, 1, 4])
def test_variance_early_stopping_inside_the_sweep(sw, idx):
    """`EarlyStopping` (reference callbacks.py:195-243: absolute change of the posterior variances)
    as the EP callback: the test runs in the sweep kernels (trb_sweep.es_mode = 1, no host round
    trip) and stops at the iteration, and in the state, of the same callback run the reference's
    way -- called on the host after every iteration."""
    from tramp_b200.algos import ExpectationPropagation, EarlyStopping, TrackEvolution, JoinCallback
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    tol = 1e-5
    runs = []
    for on_device in (True, False):
        ep = ExpectationPropagation(_build(cfg, sw, name))
        evo = TrackEvolution()
        stopper = EarlyStopping(tol=tol)
        members = [evo, stopper] if on_device else [evo, stopper, lambda algo, i, max_iter: False]
        cb = JoinCallback(members)
        assert cb.device_replayable(ep) == on_device
        ep.iterate(max_iter=200, callback=cb, damping=cfg["damping"])
        runs.append((ep.n_iter, ep.get_variables_data(), evo.get_dataframe()))
    (n_dev, d_dev, df_dev), (n_host, d_host, df_host) = runs
    assert 2 < n_dev == n_host < 200
    for vid in ("x", "z"):
        assert_allclose(d_dev[vid]["r"], d_host[vid]["r"], rtol=1e-12, atol=1e-14)
        assert_allclose(d_dev[vid]["v"], d_host[vid]["v"], rtol=1e-12)
        v = df_dev[df_dev.id == vid].v.values
        assert len(v) == n_dev and abs(v[-1] - v[-2]) < tol
        assert_allclose(v, df_host[df_host.id == vid].v.values, rtol=1e-12)


@pytest.mark.parametrize("idx", [0, 2])
def test_adaptive_schedule_device_and_host_backends_agree(ad, idx):
    """The factor-by-factor schedule kept on the device (algos/device_schedule.py: messages resident,
    objective and step-halving in kernels) against the same schedule through the numpy factor API
    (algos/factor_schedule.py): same accepted step sizes, same messages."""
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    cfg = json.loads(str(ad["configs"]))[idx]
    name = cfg["name"]
    out = {}
    for backend in ("device", "host"):
        ep = ExpectationPropagation(_build(cfg, ad, name))
        ep.schedule_backend = backend
        ep.iterate(max_iter=cfg["n_iter"], callback=PassCallback(), damping=cfg["damping"], update_dA=cfg["update_dA"])
        assert type(ep._host).__name__ == ("DeviceSchedule" if backend == "device" else "FactorSchedule")
        out[backend] = (ep.get_variables_data(), {k: dict(ep._host.edges[k]) for k in ep._host.edges}, ep.log_evidence())
    (d_dev, e_dev, A_dev), (d_host, e_host, A_host) = out["device"], out["host"]
    for vid in ("x", "z"):
        assert_allclose(d_dev[vid]["r"], d_host[vid]["r"], rtol=1e-10, atol=1e-12)
        assert_allclose(d_dev[vid]["v"], d_host[vid]["v"], rtol=1e-10)
    for k in e_host:
        assert_allclose(e_dev[k]["a"], e_host[k]["a"], rtol=1e-10)
        assert_allclose(e_dev[k]["b"], e_host[k]["b"], rtol=1e-10, atol=1e-12)
        assert e_dev[k]["n_iter"] == e_host[k]["n_iter"]
        if cfg["damping"] == "adaptive":
            assert e_dev[k]["beta"] == e_host[k]["beta"]
    assert_allclose(A_dev, A_host, rtol=1e-10)


def test_track_overlaps_and_objective_on_device_path(sw):
    """TrackOverlaps / TrackObjective are ordinary (synchronous) callbacks on the
    device path; A_model equals log_evidence()."""
    from tramp_b200.algos import ExpectationPropagation, TrackOverlaps, TrackObjective, JoinCallback
    cfg = _configs(sw)[0]
    name = cfg["name"]
    ep = ExpectationPropagation(_build(cfg, sw, name))
    x = sw[name + "_x"]
    ov, obj = TrackOverlaps({"x": x}, ids=["x"]), TrackObjective()
    ep.iterate(max_iter=cfg["n_iter"], callback=JoinCallback([ov, obj]), damping=cfg["damping"])
    df = ov.get_dataframe()
    r = ep.get_variables_data()["x"]["r"]
    assert_allclose(df.m.values[-1], r @ x / x.size, rtol=1e-12)
    assert_allclose(df.Q.values[-1], x @ x / x.size, rtol=1e-12)
    _, node_df, model_df = obj.get_dataframe()
    scale = np.abs(node_df.A.values[-5:].astype(float)).sum()
    assert abs(model_df.A.values[-1] - sw[name + "_logZ"]) <= 1e-9 * scale


def test_cuda_graph_replay_is_bitwise_identical_to_plain_launches(sw):
    """Small sweeps replay their middle iterations as a CUDA graph (trb_sweep_run);
    the kernels and their order are the same, so the results are bit-identical."""
    from tramp_b200 import _lib
    from tramp_b200.algos import ExpectationPropagation, TrackErrors
    lib = _lib.load()
    for idx in (0, 2, 4):
        cfg = _configs(sw)[idx]
        name = cfg["name"]
        out = []
        for graphs in (1, 0):
            lib.trb_set_cuda_graphs(graphs)
            lib.trb_set_persistent_sweep(0)      # the launch-per-stage path is the one under test
            try:
                ep = ExpectationPropagation(_build(cfg, sw, name))
                track = TrackErrors({"x": sw[name + "_x"]})
                lib.trb_profile_reset(0)
                ep.iterate(max_iter=cfg["n_iter"], callback=track, damping=cfg["damping"])
                d = ep.get_variables_data()
                out.append((d["x"]["r"], d["z"]["r"], d["x"]["v"], d["z"]["v"],
                            np.array([e["mse"] for e in track.errors]),
                            int(lib.trb_profile_launches(-1))))
            finally:
                lib.trb_set_cuda_graphs(1)
                lib.trb_set_persistent_sweep(-1)
        for a, b in zip(out[0][:5], out[1][:5]):
            assert np.array_equal(a, b)
        assert out[0][5] == out[1][5]      # the launch accounting counts replayed kernels too


def _sweep_with_and_without(lib, setter, on, off, build, run):
    """The same model iterated twice, with one kernel choice of trb_sweep_run switched on / off."""
    out = []
    for value in (on, off):
        getattr(lib, setter)(value)
        lib.trb_set_persistent_sweep(0)
        try:
            ep = build()
            lib.trb_profile_reset(0)
            track = run(ep)
            d = ep.get_variables_data()
            out.append(dict(rx=d["x"]["r"], rz=d["z"]["r"], vx=d["x"]["v"], vz=d["z"]["v"],
                            mse=np.array([e["mse"] for e in track.errors]),
                            n_iter=np.array(ep.n_iter_per_instance),
                            launches=int(lib.trb_profile_launches(-1))))
        finally:
            getattr(lib, setter)(on)
            lib.trb_set_persistent_sweep(-1)
    assert np.array_equal(out[0]["n_iter"], out[1]["n_iter"])
    return out


def _kernel_choice_cases(sw):
    """(build, run) pairs: single instances spread over many CTAs (golden configs) and a batch
    whose instances stop at different iterations."""
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import ExpectationPropagation, TrackErrors, EarlyStoppingEP, JoinCallback
    cases = []
    for idx in (0, 2, 4, 6):
        cfg = _configs(sw)[idx]
        name = cfg["name"]

        def run(ep, cfg=cfg, name=name):
            track = TrackErrors({"x": sw[name + "_x"]})
            ep.iterate(max_iter=cfg["n_iter"], callback=track, damping=cfg["damping"])
            return track
        cases.append((lambda cfg=cfg, name=name: ExpectationPropagation(_build(cfg, sw, name)), run, False))
    rng = np.random.RandomState(19)
    B, N, M = 7, 2500, 1300            # three chunks of x, two of z per instance
    W = rng.randn(B, M, N) / np.sqrt(N)
    x = rng.randn(B, N) * (rng.rand(B, N) < 0.1)
    y = np.einsum("bmn,bn->bm", W, x) + 0.1 * rng.randn(B, M)
    lin = LinearChannel(W)
    lin._setup()                       # factorise once, outside the launch counts

    def build():
        return ExpectationPropagation((GaussBernoulliPrior(size=N, rho=0.1, batch=B) @ V("x") @ lin @ V("z")
                                       @ GaussianLikelihood(y=y, var=1e-2)).to_model())

    def run_es(ep):
        track = TrackErrors({"x": x})
        ep.schedule = "general"
        ep.iterate(max_iter=200, callback=JoinCallback([track, EarlyStoppingEP(tol=1e-6)]))
        return track
    cases.append((build, run_es, True))
    # rows wider than one stage of the TMA ring: the projection of V walks two column panels and
    # the coefficient is written with the last one
    B2, N2, M2 = 2, 8300, 48
    W2 = rng.randn(B2, M2, N2) / np.sqrt(N2)
    x2 = rng.randn(B2, N2) * (rng.rand(B2, N2) < 0.05)
    y2 = np.einsum("bmn,bn->bm", W2, x2) + 0.1 * rng.randn(B2, M2)
    lin2 = LinearChannel(W2)
    lin2._setup()

    def build2():
        return ExpectationPropagation((GaussBernoulliPrior(size=N2, rho=0.05, batch=B2) @ V("x") @ lin2 @ V("z")
                                       @ GaussianLikelihood(y=y2, var=1e-2)).to_model())

    def run2(ep):
        track = TrackErrors({"x": x2})
        ep.schedule = "general"
        ep.iterate(max_iter=12, callback=track, damping=0.1)
        return track
    cases.append((build2, run2, False))
    return cases


def test_rescale_inside_the_projection_equals_separate_launches(sw):
    """trb_sweep_run runs the rescale stages S1 / S2 inside the GEMV projections P1 / P3 (the
    thread that finishes a row's block reduction writes the row's coefficient; the CTA that owns
    an instance's first row computes the variance).  Same arithmetic per coefficient; only the
    order of the spectrum sum behind the variance differs: 1e-12 against the nine-launch
    iteration, with two launches fewer per iteration."""
    from tramp_b200 import _lib
    lib = _lib.load()
    for build, run, batch in _kernel_choice_cases(sw):
        a, b = _sweep_with_and_without(lib, "trb_set_fused_rescale", 1, 0, build, run)
        for k in ("rx", "rz", "vx", "vz", "mse"):       # mse: NaN once an instance has stopped
            assert_allclose(a[k], b[k], rtol=1e-12, atol=1e-12 * np.nanmax(np.abs(b[k])), err_msg=k)
        assert a["launches"] < b["launches"]
        if batch:
            assert len(set(a["n_iter"].tolist())) > 1     # the instances did stop at different iterations


def test_chunked_update_kernels_equal_one_cta_per_instance(sw):
    """trb_set_update_kernels: the chunked x / z updates (1024 elements per CTA, the last-arriving
    CTA adds the chunk sums) do the arithmetic of k_x_update / k_z_update element for element:
    messages and posteriors are bit-identical; only the sums behind the recorded mse / tolerance
    are added in another order."""
    from tramp_b200 import _lib
    lib = _lib.load()
    for build, run, batch in _kernel_choice_cases(sw):
        for mask in (1, 2, 3):
            a, b = _sweep_with_and_without(lib, "trb_set_update_kernels", mask, 0, build, run)
            lib.trb_set_update_kernels(-1)
            for k in ("rx", "rz", "vx", "vz"):
                assert np.array_equal(a[k], b[k]), (mask, k)
            assert_allclose(a["mse"], b["mse"], rtol=1e-12)
            assert a["launches"] == b["launches"]


@pytest.mark.parametrize("idx", range(9))
def test_persistent_sweep_matches_launch_per_stage_path(sw, idx):
    """One instance runs all its iterations inside ONE launch (trb_persist.cu, four
    barriers per iteration): as a cooperative grid of one CTA per SM (mode 2) or,
    for the smallest instances, as a single 16-CTA cluster with the hardware
    cluster barrier (mode 3).  Same arithmetic per element, different summation
    order in the operator passes: 1e-11 against the launch-per-stage path (mode
    0), and the golden vectors of the reference at 1e-9."""
    from tramp_b200 import _lib
    from tramp_b200.algos import ExpectationPropagation, TrackErrors, TrackEvolution, JoinCallback
    lib = _lib.load()
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    out = {}
    for mode in (3, 2, 0):
        lib.trb_set_persistent_sweep(mode)
        try:
            ep = ExpectationPropagation(_build(cfg, sw, name))
            ep.schedule = "general"
            track = TrackErrors({"x": sw[name + "_x"]}, metrics=["mse", "sign_mse"])
            evo = TrackEvolution()
            init = _SeqInit(sw, name) if cfg.get("init") == "noisy" else None
            ep.linear._setup()             # the factorisation's launches are not the sweep's
            lib.trb_profile_reset(0)
            ep.iterate(max_iter=cfg["n_iter"], callback=JoinCallback([track, evo]), initializer=init,
                       damping=cfg["damping"])
            launches = int(lib.trb_profile_launches(-1))
            d = ep.get_variables_data()
            df = evo.get_dataframe()
            out[mode] = dict(rx=d["x"]["r"], rz=d["z"]["r"], vx=d["x"]["v"], vz=d["z"]["v"],
                             mse=np.array([e["mse"] for e in track.errors]),
                             smse=np.array([e["sign_mse"] for e in track.errors]),
                             vxt=df[df.id == "x"].v.values, vzt=df[df.id == "z"].v.values,
                             edges=[ep._edge(f"e{k}") for k in range(1, 9)], n_iter=ep.n_iter,
                             launches=launches)
        finally:
            lib.trb_set_persistent_sweep(-1)
    q = out[0]
    assert q["launches"] >= 5 * cfg["n_iter"]          # launch-per-stage path: at least F1, P1..P4 per iteration
    x, W = sw[name + "_x"], sw[name + "_W"]
    tau_x, tau_z = np.mean(x**2), np.mean((W @ x)**2)
    saturated = max(float(sw[f"{name}_e{k}_a"]) for k in range(1, 9)) > 1e4
    tol = 1e-9 if saturated else 1e-11          # ill-conditioned at exact recovery, see DESIGN "Parity"
    for mode in (3, 2):
        p = out[mode]
        assert p["launches"] == 1
        assert p["n_iter"] == q["n_iter"] == cfg["n_iter"]
        for key, scale in (("rx", np.abs(q["rx"]).max()), ("rz", np.abs(q["rz"]).max()), ("vx", tau_x),
                           ("vz", tau_z), ("vxt", tau_x), ("vzt", tau_z)):
            assert_allclose(p[key], q[key], rtol=tol, atol=tol * scale)
        for key in ("mse", "smse"):
            assert np.all(np.abs(p[key] - q[key]) <= tol * q[key] + 2 * tol * np.sqrt(q[key] * tau_x))
        if not saturated:
            for (a1, b1), (a0, b0) in zip(p["edges"], q["edges"]):
                assert_allclose(a1, a0, rtol=tol)
                assert_allclose(b1, b0, rtol=tol, atol=tol * np.abs(b0).max())
        # and the reference itself
        ref = sw[name + "_mse"]
        assert np.all(np.abs(p["mse"] - ref) <= 1e-9 * ref + 2e-9 * np.sqrt(ref * tau_x))
        ref = sw[name + "_rx"]
        assert_allclose(p["rx"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
        assert_allclose(p["vx"], sw[name + "_vx_final"], rtol=1e-9, atol=1e-9 * tau_x)


@pytest.mark.parametrize("mode", [2, 3])
def test_persistent_sweep_early_stopping_rollback_and_warm_start(sw, mode):
    """The persistent kernel (grid and cluster variants) takes the same
    EarlyStoppingEP decisions (convergence, divergence with roll-back to the
    previous iteration), leaves live / snapshot buffers consistent for a warm
    start, and reports NaN like the other path."""
    from tramp_b200 import _lib
    from tramp_b200.algos import ExpectationPropagation, PassCallback
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    lib = _lib.load()
    lib.trb_set_persistent_sweep(mode)
    try:
        for idx in range(3):                                   # convergence at the reference's iteration
            cfg = _configs(sw)[idx]
            name = cfg["name"] + "_early"
            ep = ExpectationPropagation(_build(cfg, sw, name))
            ep.iterate(max_iter=200, damping=cfg["damping"])
            assert ep.n_iter == int(sw[name + "_n_iter"])
            ref = sw[name + "_rx"]
            assert_allclose(ep.get_variables_data()["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
        name = "cs_diverges_early"                             # divergence: rolled back
        model = (GaussBernoulliPrior(size=120, rho=0.1) @ V("x") @ LinearChannel(sw[name + "_W"])
                 @ V("z") @ GaussianLikelihood(y=sw[name + "_y"], var=1e-2)).to_model()
        ep = ExpectationPropagation(model)
        ep.iterate(max_iter=200)
        assert ep.n_iter == int(sw[name + "_n_iter"]) == 7
        d = ep.get_variables_data()
        assert_allclose(d["x"]["r"], sw[name + "_rx"], rtol=1e-9, atol=1e-12)
        assert_allclose(d["z"]["r"], sw[name + "_rz"], rtol=1e-9, atol=1e-12)
        for k in range(1, 9):
            a, b = ep._edge(f"e{k}")
            assert_allclose(a, sw[f"{name}_e{k}_a"], rtol=1e-9)
            assert_allclose(b, sw[f"{name}_e{k}_b"], rtol=1e-9, atol=1e-12)
        cfg = _configs(sw)[0]                                  # odd + even splits of a warm-started run
        name = cfg["name"]
        ep = ExpectationPropagation(_build(cfg, sw, name))
        ep.iterate(max_iter=7, callback=PassCallback())
        ep.iterate(max_iter=8, callback=PassCallback(), warm_start=True)
        ep.iterate(max_iter=cfg["n_iter"] - 15, callback=PassCallback(), warm_start=True)
        assert ep.n_iter == cfg["n_iter"]
        ref = sw[name + "_rx"]
        assert_allclose(ep.get_variables_data()["x"]["r"], ref, rtol=1e-9, atol=1e-9 * np.abs(ref).max())
        y_bad = sw[name + "_y"].copy()                         # NaN surfaces as ValueError
        y_bad[3] = np.nan
        from tramp_b200.priors import get_prior
        from tramp_b200.likelihoods import get_likelihood
        pk = {k: v for k, v in cfg["prior"].items() if k != "kind"}
        lk = {k: v for k, v in cfg["lik"].items() if k != "kind"}
        bad = (get_prior(size=cfg["N"], prior_type=cfg["prior"]["kind"], **pk) @ V("x")
               @ LinearChannel(sw[name + "_W"]) @ V("z")
               @ get_likelihood(y=y_bad, likelihood_type=cfg["lik"]["kind"], **lk)).to_model()
        with pytest.raises(ValueError, match="nan"):
            ExpectationPropagation(bad).iterate(max_iter=5, callback=PassCallback())
    finally:
        lib.trb_set_persistent_sweep(-1)


@pytest.mark.parametrize("lik_kind", ["gaussian", "sgn"])
def test_cluster_split_update_kernels_match_one_cta_per_instance(lik_kind):
    """A single large instance spreads its per-instance update kernels over a
    thread-block cluster (DSMEM reductions, trb_cluster_size > 1); the same
    instance inside a batch that fills the GPU uses one CTA per instance.  Same
    arithmetic, different summation order: agreement to ~1e-12."""
    import torch
    from tramp_b200 import synthetic
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood, SgnLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import ExpectationPropagation, TrackErrors
    N, M, n_iter, Bbig = 16384, 8192, 12, 80
    data = synthetic.gaussian_glm_batch(1, N, M, rho=0.1, var_noise=1e-2, seed=3, chunk=1, workers=1)
    y = data["y"] if lik_kind == "gaussian" else torch.where(data["z"] >= 0, 1.0, -1.0).to(torch.float64)
    outs = []
    for B in (1, Bbig):
        lin = LinearChannel.from_factors(data["Ut"], data["s"], data["Vt"], Nx=M, Nz=N, rank=M)
        yb = y if B == 1 else y.expand(B, M).contiguous()
        lik = (GaussianLikelihood(y=yb[0] if B == 1 else yb, var=1e-2) if lik_kind == "gaussian"
               else SgnLikelihood(y=yb[0] if B == 1 else yb))
        prior = GaussBernoulliPrior(size=N, rho=0.1) if B == 1 else GaussBernoulliPrior(size=N, rho=0.1, batch=B)
        ep = ExpectationPropagation((prior @ V("x") @ lin @ V("z") @ lik).to_model())
        ep.linear_backend = "gemv"        # keep the GEMV passes for the batch too (shared operator)
        ep.schedule = "general"
        xt = data["x"][0] if B == 1 else data["x"].expand(B, N).contiguous()
        track = TrackErrors({"x": xt})
        ep.iterate(max_iter=n_iter, callback=track, damping=0.2)
        d = ep.get_variables_data()
        pick = (lambda a: a) if B == 1 else (lambda a: a[0])
        outs.append((pick(d["x"]["r"]), pick(d["z"]["r"]), pick(d["x"]["v"]), pick(d["z"]["v"]),
                     np.array([pick(e["mse"]) for e in track.errors])))
    from tramp_b200 import _lib
    assert _lib.load().trb_device_sm_count() > 0
    for a, b in zip(*outs):
        assert_allclose(a, b, rtol=1e-10, atol=1e-12 * max(1.0, np.abs(b).max()))
    assert outs[0][4][-1] < outs[0][4][0]          # EP made progress
