"""Pin the CPU oracle (oracle/tramp_oracle.py) against the golden vectors that
tests/golden/make_golden.py produced from the unmodified reference."""
import json
import os
import numpy as np
import pytest
from numpy.testing import assert_allclose

from oracle import tramp_oracle as orc
from tests.golden import load_sweeps
from tests.golden.make_golden_specs import PRIOR_SPECS, LIK_SPECS, TRUNC_CASES

RTOL = 1e-12


@pytest.fixture(scope="module")
def el(golden_dir):
    return np.load(os.path.join(golden_dir, "elementwise.npz"))


@pytest.fixture(scope="module")
def lin(golden_dir):
    return np.load(os.path.join(golden_dir, "linear.npz"))


@pytest.fixture(scope="module")
def sw(golden_dir):
    return load_sweeps(golden_dir)


@pytest.mark.parametrize("i", range(len(PRIOR_SPECS)))
def test_prior_elementwise(el, i):
    spec = dict(PRIOR_SPECS[i], isotropic=False)
    a, b = el["grid_a"], el["grid_b"]
    with np.errstate(all="ignore"):
        r, v = orc.prior_forward_posterior(spec, a, b)
    assert_allclose(r, el[f"prior{i}_r"], rtol=RTOL, atol=1e-300)
    assert_allclose(v * np.ones_like(a), el[f"prior{i}_v"], rtol=RTOL, atol=1e-300)
    for j, a_s in enumerate(el["iso_a"]):
        spec = dict(PRIOR_SPECS[i], isotropic=True)
        b = el["grid_bnorm"] * np.sqrt(a_s)
        r, v = orc.prior_forward_posterior(spec, a_s, b)
        an, bn = orc.prior_forward_message(spec, a_s, b)
        assert_allclose(r, el[f"prior{i}_iso{j}_r"], rtol=RTOL, atol=1e-300)
        assert_allclose(v, el[f"prior{i}_iso{j}_v"], rtol=RTOL)
        assert_allclose(an, el[f"prior{i}_iso{j}_anew"], rtol=RTOL)
        assert_allclose(bn * np.ones_like(b), el[f"prior{i}_iso{j}_bnew"], rtol=RTOL, atol=1e-300)
        A = orc.prior_log_partition(spec, a_s, b)
        assert_allclose(A, el[f"prior{i}_iso{j}_A"], rtol=RTOL)


@pytest.mark.parametrize("i", range(len(LIK_SPECS)))
def test_likelihood_elementwise(el, i):
    a, b = el["grid_a"], el["grid_b"]
    y = el[f"lik{i}_y"]
    spec = dict(LIK_SPECS[i], y=y, isotropic=False)
    with np.errstate(all="ignore"):
        r, v = orc.likelihood_backward_posterior(spec, a, b)
    assert_allclose(r, el[f"lik{i}_r"], rtol=RTOL, atol=1e-300)
    assert_allclose(v * np.ones_like(a), el[f"lik{i}_v"], rtol=RTOL, atol=1e-300)
    for j, a_s in enumerate(el["iso_a"]):
        spec = dict(LIK_SPECS[i], y=y, isotropic=True)
        b = el["grid_bnorm"] * np.sqrt(a_s)
        r, v = orc.likelihood_backward_posterior(spec, a_s, b)
        an, bn = orc.likelihood_backward_message(spec, a_s, b)
        assert_allclose(r, el[f"lik{i}_iso{j}_r"], rtol=RTOL, atol=1e-300)
        assert_allclose(v, el[f"lik{i}_iso{j}_v"], rtol=RTOL)
        assert_allclose(an, el[f"lik{i}_iso{j}_anew"], rtol=RTOL)
        assert_allclose(bn * np.ones_like(b), el[f"lik{i}_iso{j}_bnew"], rtol=RTOL, atol=1e-300)
        A = orc.likelihood_log_partition(spec, a_s, b)
        assert_allclose(A, el[f"lik{i}_iso{j}_A"], rtol=RTOL)


@pytest.mark.parametrize("i", range(len(TRUNC_CASES)))
def test_truncated_beliefs(el, i):
    a, lo, hi = TRUNC_CASES[i]
    b = el["trunc_b"]
    with np.errstate(all="ignore"):
        assert_allclose(orc.truncated_A(a, b, lo, hi), el[f"trunc{i}_A"], rtol=RTOL, equal_nan=True)
        assert_allclose(orc.truncated_r(a, b, lo, hi), el[f"trunc{i}_r"], rtol=RTOL, equal_nan=True)
        assert_allclose(orc.truncated_v(a, b, lo, hi), el[f"trunc{i}_v"], rtol=RTOL, atol=1e-300, equal_nan=True)
        assert_allclose(orc.truncated_p(a, b, lo, hi), el[f"trunc{i}_p"], rtol=RTOL, atol=1e-300, equal_nan=True)


def test_positive_beliefs(el):
    a, b = el["pos_a"], el["pos_b"]
    assert_allclose(orc.positive_A(a, b), el["pos_A"], rtol=RTOL)
    assert_allclose(orc.positive_r(a, b), el["pos_r"], rtol=RTOL)
    assert_allclose(orc.positive_v(a, b), el["pos_v"], rtol=RTOL, atol=1e-300)


def test_linear_channel(lin):
    for i in range(int(lin["lin_nW"])):
        op = orc.LinearOp(lin[f"lin{i}_W"])
        assert op.rank == int(lin[f"lin{i}_rank"])
        bz, bx = lin[f"lin{i}_bz"], lin[f"lin{i}_bx"]
        for j, (az, ax) in enumerate(lin["lin_ab"]):
            with np.errstate(all="ignore"):
                rz, vz = orc.lin_backward_posterior(op, az, bz, ax, bx)
                A = orc.lin_log_partition(op, az, bz, ax, bx)
                assert_allclose(orc.lin_n_eff(op, az, ax), lin[f"lin{i}_{j}_neff"], rtol=RTOL)
            assert_allclose(rz, lin[f"lin{i}_{j}_rz"], rtol=1e-10, atol=1e-12, equal_nan=True)
            assert_allclose(vz, lin[f"lin{i}_{j}_vz"], rtol=RTOL, equal_nan=True)
            assert_allclose(A, lin[f"lin{i}_{j}_A"], rtol=1e-10, equal_nan=True)
            if az > 0:
                rx, vx = orc.lin_forward_posterior(op, az, bz, ax, bx)
                assert_allclose(rx, lin[f"lin{i}_{j}_rx"], rtol=1e-10, atol=1e-12)
                assert_allclose(vx, lin[f"lin{i}_{j}_vx"], rtol=RTOL)


def _configs(sw):
    return json.loads(str(sw["configs"]))


def _init_from(sw, name):
    if f"{name}_init_e1_a" not in sw:
        return None
    return {f"e{k}": (float(sw[f"{name}_init_e{k}_a"]), sw[f"{name}_init_e{k}_b"])
            for k in range(1, 9)}


@pytest.mark.parametrize("idx", range(9))
def test_sweep_fixed_iterations(sw, idx):
    cfg = _configs(sw)[idx]
    name = cfg["name"]
    lik = dict(cfg["lik"], y=sw[name + "_y"])
    with np.errstate(all="ignore"):
        out = orc.ep_glm(cfg["prior"], sw[name + "_W"], lik, cfg["n_iter"],
                         damping=cfg["damping"], init=_init_from(sw, name),
                         x_true=sw[name + "_x"])
    tol = dict(rtol=1e-9, atol=1e-12)
    assert_allclose(out["traj"]["mse_x"], sw[name + "_mse"], rtol=1e-9, atol=1e-30)
    assert_allclose(out["traj"]["v_x"], sw[name + "_vx"], rtol=1e-9)
    assert_allclose(out["traj"]["v_z"], sw[name + "_vz"], rtol=1e-9)
    assert_allclose(out["r_x"], sw[name + "_rx"], **tol)
    assert_allclose(out["r_z"], sw[name + "_rz"], **tol)
    for k in range(1, 9):
        a, b = out["edges"][f"e{k}"]
        assert_allclose(a, sw[f"{name}_e{k}_a"], rtol=1e-9)
        assert_allclose(b, sw[f"{name}_e{k}_b"], rtol=1e-9,
                        atol=1e-9 * np.abs(sw[f"{name}_e{k}_b"]).max())
    with np.errstate(all="ignore"):
        logZ, parts = orc.ep_log_evidence(cfg["prior"], out["op"], lik, out["edges"])
    assert_allclose(logZ, sw[name + "_logZ"], rtol=1e-8)


@pytest.mark.parametrize("idx", range(3))
def test_sweep_early_stopping(sw, idx):
    cfg = _configs(sw)[idx]
    name = cfg["name"] + "_early"
    lik = dict(cfg["lik"], y=sw[name + "_y"])
    out = orc.ep_glm(cfg["prior"], sw[name + "_W"], lik, 200, damping=cfg["damping"],
                     early_stopping=dict(tol=1e-6))
    assert out["n_iter"] == int(sw[name + "_n_iter"])
    assert out["status"] == "converged"
    assert_allclose(out["r_x"], sw[name + "_rx"], rtol=1e-9, atol=1e-12)
    assert_allclose(out["v_x"], sw[name + "_vx_final"], rtol=1e-9)


def test_sweep_early_stopping_divergence_branch(sw):
    """EarlyStoppingEP's max_increase branch: messages and estimates roll back one iteration."""
    name = "cs_diverges_early"
    lik = dict(kind="gaussian", var=1e-2, y=sw[name + "_y"])
    out = orc.ep_glm(dict(kind="gauss_bernoulli", rho=0.1), sw[name + "_W"], lik, 200,
                     early_stopping=dict(tol=1e-6))
    assert out["status"] == "diverged" and out["n_iter"] == int(sw[name + "_n_iter"]) == 7
    assert_allclose(out["r_x"], sw[name + "_rx"], rtol=1e-9, atol=1e-12)
    assert_allclose(out["r_z"], sw[name + "_rz"], rtol=1e-9, atol=1e-12)
    assert_allclose(out["v_x"], sw[name + "_vx_final"], rtol=1e-9)
    for k in range(1, 9):
        assert_allclose(out["edges"][f"e{k}"][0], sw[f"{name}_e{k}_a"], rtol=1e-9)
        assert_allclose(out["edges"][f"e{k}"][1], sw[f"{name}_e{k}_b"], rtol=1e-9, atol=1e-12)
