"""The bodies of the GPU API tests (tests/test_gpu_api.py) run in the build container
through the emulated device (tests/_emulated_device.py): the sweep by the oracle, the
per-factor primitives by the device moment routines compiled for the host and numpy.

What this covers on CPU: every Python layer between the public API and the C ABI --
the factor API of priors / likelihoods / LinearChannel and the beliefs wrappers (the
reference's own unit tests, tramp/tests/test_{beliefs,priors,likelihoods}.py), the
host-driven factor-by-factor schedule of `damping="adaptive"` / `update_dA` against the
reference's golden runs, the log-evidence assembly, callbacks on both iteration paths,
warm starts, early stopping per instance, the Gram set-up, scenarios.  The kernels
themselves are what the same tests check on the GPU.

Left to the GPU only: tests that select kernel variants (GEMV implementations,
persistent / CUDA-graph / cluster shapes, DMMA and cuBLAS back ends)."""
import os

import numpy as np
import pytest

from tests._emulated_device import emulated_device  # noqa: F401  (fixture)
from tests import test_gpu_api as G
from tests.golden import load_sweeps


@pytest.fixture(scope="module")
def sw(golden_dir):
    return load_sweeps(golden_dir)


@pytest.fixture(scope="module")
def ad(golden_dir):
    return np.load(os.path.join(golden_dir, "adaptive.npz"))


def test_factor_api_mirrors_reference_unit_tests(emulated_device):  # noqa: F811
    G.test_factor_api_mirrors_reference_unit_tests()


def test_belief_gradients(emulated_device):  # noqa: F811
    G.test_belief_gradients()


def test_beliefs_against_reference(emulated_device, golden_dir):  # noqa: F811
    G.test_beliefs_against_reference(golden_dir)


@pytest.mark.parametrize("idx", [0, 1, 4])
def test_variance_early_stopping_inside_the_sweep(emulated_device, sw, idx):  # noqa: F811
    G.test_variance_early_stopping_inside_the_sweep(sw, idx)


def test_noisy_init_consumes_the_random_stream_like_the_reference(emulated_device, sw):  # noqa: F811
    G.test_noisy_init_consumes_the_random_stream_like_the_reference(sw)


def test_linear_channel_reference_signature_corners(emulated_device):  # noqa: F811
    G.test_linear_channel_reference_signature_corners()


def test_linear_channel_factor_api(emulated_device, golden_dir):  # noqa: F811
    G.test_linear_channel_factor_api(golden_dir)


@pytest.mark.parametrize("idx", range(4))
def test_adaptive_damping_and_dA_match_reference(emulated_device, ad, idx):  # noqa: F811
    G.test_adaptive_damping_and_dA_match_reference(ad, idx)


@pytest.mark.parametrize("idx", [0, 2])
def test_adaptive_schedule_device_and_host_backends_agree(emulated_device, ad, idx):  # noqa: F811
    G.test_adaptive_schedule_device_and_host_backends_agree(ad, idx)


def test_host_path_then_device_warm_start(emulated_device, ad):  # noqa: F811
    G.test_host_path_then_device_warm_start(ad)


@pytest.mark.parametrize("options", [dict(damping="adaptive"), dict(damping=0.2, update_dA=True)])
def test_adaptive_damping_batched_equals_per_instance(emulated_device, options):  # noqa: F811
    G.test_adaptive_damping_batched_equals_per_instance(options)


@pytest.mark.parametrize("idx", range(9))
def test_sweep_matches_reference(emulated_device, sw, idx):  # noqa: F811
    G.test_sweep_matches_reference(sw, idx, 2, "auto")


@pytest.mark.parametrize("idx", range(9))
def test_log_evidence_matches_reference(emulated_device, sw, idx):  # noqa: F811
    G.test_log_evidence_matches_reference(sw, idx)


@pytest.mark.parametrize("idx", range(3))
def test_default_early_stopping(emulated_device, sw, idx):  # noqa: F811
    G.test_default_early_stopping(sw, idx)


@pytest.mark.parametrize("name", ["test_early_stopping_divergence_restores_previous_iteration",
                                  "test_synchronous_callback_path_equals_device_path",
                                  "test_warm_start_continues", "test_errors_mirror_reference",
                                  "test_track_overlaps_and_objective_on_device_path"])
def test_driver_paths(emulated_device, sw, name):  # noqa: F811
    getattr(G, name)(sw)


def test_batched_early_stopping_per_instance(emulated_device):  # noqa: F811
    G.test_batched_early_stopping_per_instance()


@pytest.mark.parametrize("idx", [0, 2, 5])
def test_gram_factorisation_matches_reference(emulated_device, sw, idx):  # noqa: F811
    G.test_gram_factorisation_matches_reference(sw, idx)


def test_scenario_and_glm_generative(emulated_device):  # noqa: F811
    G.test_scenario_and_glm_generative()


def test_emulated_linear_primitives_follow_the_kernels(emulated_device, golden_dir):  # noqa: F811
    """project -> rescale -> expand against the golden LinearChannel vectors
    (tests/test_gpu_primitives.py): pins the numpy restatement of k_lin_rescale /
    the slot reduction that the emulation above relies on."""
    from tests import test_gpu_primitives as P
    from tramp_b200 import ops
    P.test_linear_channel_primitives(ops, np.load(os.path.join(golden_dir, "linear.npz")), 1)
