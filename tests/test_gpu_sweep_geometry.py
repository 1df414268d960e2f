"""The EP sweep against the float64 oracle on both sides of every shape-dependent kernel choice
of trb_sweep_run: the tile width NB of the TMA GEMVs (and their column panels), the expansion
slots per instance, the 32- / 64-bit slot arithmetic, the chunks of the x / z updates, the
cluster size of the per-instance updates, the persistent kernel's variants and fall-backs, the
shared-operator back ends and the shape / rank of W.

Every row names the decision it is meant to land on, is compared with `oracle.ep_glm` at 1e-9
(the tolerance rules of tests/test_gpu_api.py::test_sweep_matches_reference), and proves from a
torch.profiler trace that the kernels of that decision ran.  The oracle takes a full SVD; for
operators with max(M, N) > 10000 its linear-channel means are replaced by `DenseLinear`, which
needs W only.  The last test asserts that the rows together reached every decision value."""
import contextlib
import json
import re

import numpy as np
import pytest

from oracle import tramp_oracle as orc

N_ITER = 8
SEEN = dict(kernels=set(), clusters=set(), ns=set(), slots_word=set())


# ---------------------------------------------------------------- dense reference
class DenseLinear:
    """The LinearChannel of the oracle without an SVD: the means solve the smaller of the two
    Gram systems, the spectrum the variances need is the eigenvalues of the smaller Gram matrix.
    Same attribute names as oracle.LinearOp, so the oracle's variance functions take it as is."""

    AMIN, AMAX = orc.AMIN, orc.AMAX

    def __init__(self, W):
        W = np.asarray(W, dtype=float)
        self.W = W
        self.Nx, self.Nz = W.shape
        self.alpha = self.Nx / self.Nz
        self.tall = self.Nx >= self.Nz
        self.G = W.T @ W if self.tall else W @ W.T
        self.rank = np.linalg.matrix_rank(W)          # linear_channel.py:37 (singular values only)
        self.singular = np.linalg.eigvalsh(self.G)[::-1][:self.rank]

    def backward_mean(self, az, bz, ax, bx):
        """(az I + ax W^T W)^-1 (bz + W^T bx): linear_channel.py:69-83 without the SVD."""
        v = bz + self.W.T @ bx
        if self.tall:
            return np.linalg.solve(az * np.eye(self.Nz) + ax * self.G, v)
        # Woodbury: (1/az) (I - ax W^T (az I_M + ax W W^T)^-1 W)
        return (v - ax * (self.W.T @ np.linalg.solve(az * np.eye(self.Nx) + ax * self.G, self.W @ v))) / az


@contextlib.contextmanager
def _dense_means():
    orig = orc.lin_backward_mean

    def backward_mean(op, az, bz, ax, bx):
        if isinstance(op, DenseLinear):
            return op.backward_mean(az, bz, ax, bx)
        return orig(op, az, bz, ax, bx)
    orc.lin_backward_mean = backward_mean
    try:
        yield
    finally:
        orc.lin_backward_mean = orig


def _ref_op(W):
    return DenseLinear(W) if max(W.shape) > 10000 else orc.LinearOp(W)


def test_dense_reference_equals_svd_reference():
    """DenseLinear against oracle.LinearOp on small tall, wide, square and rank-deficient W:
    channel means and variances, and a whole oracle EP run."""
    rng = np.random.RandomState(11)
    for M, N in ((30, 20), (20, 30), (25, 25), (18, 27)):
        W = rng.randn(M, N) / np.sqrt(N)
        if (M, N) == (18, 27):
            W[1] = W[0]
        full, dense = orc.LinearOp(W), DenseLinear(W)
        assert dense.rank == full.rank
        for az, ax in ((1.3, 0.0), (0.7, 2.1), (1e-3, 1e3), (40.0, 1e-2)):
            bz, bx = rng.randn(N), rng.randn(M)
            with _dense_means():
                (r1, v1), (r0, v0) = (orc.lin_backward_posterior(op, az, bz, ax, bx) for op in (dense, full))
                np.testing.assert_allclose(r1, r0, rtol=1e-11, atol=1e-11 * np.abs(r0).max())
                np.testing.assert_allclose(v1, v0, rtol=1e-12)
                # W rz cancels where ax s^2 >> az: rounding relative to |W| |rz|, not to the result
                (f1, v1), (f0, v0) = (orc.lin_forward_posterior(op, az, bz, ax, bx) for op in (dense, full))
                np.testing.assert_allclose(f1, f0, rtol=0, atol=1e-11 * (np.abs(W) @ np.abs(r0)).max())
                np.testing.assert_allclose(v1, v0, rtol=1e-12)
        x = rng.randn(N) * (rng.rand(N) < 0.3)
        y = W @ x + 0.1 * rng.randn(M)
        prior, lik = dict(kind="gauss_bernoulli", rho=0.3), dict(kind="gaussian", var=0.01, y=y)
        with _dense_means():
            a = orc.ep_glm(prior, W, lik, 10, damping=0.2, x_true=x, op=dense)
        b = orc.ep_glm(prior, W, lik, 10, damping=0.2, x_true=x, op=full)
        for k in ("r_x", "r_z"):
            np.testing.assert_allclose(a[k], b[k], rtol=1e-10, atol=1e-10 * np.abs(b[k]).max())
        np.testing.assert_allclose(a["traj"]["mse_x"], b["traj"]["mse_x"], rtol=1e-10)


def test_sweep_rejects_more_instances_than_grid_rows():
    """Every per-instance launch of the sweep puts the instance in gridDim.y (<= 65535): a
    descriptor with more instances is refused by the shape check, before any launch."""
    import ctypes as C
    from tramp_b200 import _lib
    lib = _lib.load()
    sw = _lib.TrbSweep()
    sw.B, sw.N, sw.M, sw.R = 70000, 64, 64, 64       # no buffers: the shape check comes first
    assert lib.trb_sweep_run(C.byref(sw), 0, 1, 0, None) != 0
    assert b"B > 65535" in lib.trb_last_error()
    assert lib.trb_sweep_stage(C.byref(sw), 0, 0, 0, 0, None) != 0
    assert b"B > 65535" in lib.trb_last_error()


# ---------------------------------------------------------------- case table
def _case(cid, N, M, B=1, prior="gauss_bernoulli", lik="gaussian", damping=0.3, schedule="general",
          shared=False, backend=None, persist=0, fused=1, upd=-1, rankdef=False, patterns=None,
          n_iter=N_ITER, expect=(), absent=(), decision=None, ref=None):
    """One row.  persist / fused / upd: trb_set_persistent_sweep / _fused_rescale /
    _update_kernels for the run.  expect: (kernel regex, grid.x or None) that must appear in the
    trace; absent: kernel regexes that must not.  patterns: the instances repeat this many
    distinct problems (big batches).  ref: the key of the oracle run (rows that differ only in a
    kernel switch share it)."""
    return pytest.param(dict(id=cid, N=N, M=M, B=B, prior=prior, lik=lik, damping=damping,
                             schedule=schedule, shared=shared, backend=backend, persist=persist,
                             fused=fused, upd=upd, rankdef=rankdef, patterns=patterns, n_iter=n_iter,
                             expect=list(expect), absent=list(absent), decision=decision or {},
                             ref=ref or cid), id=cid)


# ld = N padded to 16 doubles; NB = column pairs per consumer thread (ld / 512, rounded up to a
# power of two); ld > 8192: column panels of NB = 16
_WIDTHS = ((512, 1), (513, 2), (1024, 2), (1025, 4), (2048, 4), (2049, 8), (4096, 8), (4097, 16),
           (8192, 16), (8193, 16))
GEMV_CASES = []
for _w, _nb in _WIDTHS:
    for _fused in (1, 0):
        _modes = ((2, 1) if _fused else (0, 1))
        _extra = () if _fused else (("k_lin_rescale", None),)
        # N = w: V's passes (P1 project, P4 expand); M = 48 keeps U's at NB = 1
        GEMV_CASES.append(_case(f"gemv_N{_w}_fused{_fused}", N=_w, M=48, fused=_fused, ref=f"gemv_N{_w}",
                                expect=[(f"k_gemv_tma<{_nb},{m}>", None) for m in _modes] + list(_extra),
                                decision=dict(nb=_nb, side="V")))
        # M = w: U's passes (P2 expand, P3 project), sgn likelihood (k_z_update)
        GEMV_CASES.append(_case(f"gemv_M{_w}_fused{_fused}", N=40, M=_w, prior="gaussian", lik="sgn",
                                fused=_fused, ref=f"gemv_M{_w}",
                                expect=[(f"k_gemv_tma<{_nb},{m}>", None) for m in _modes] + list(_extra)
                                + [("k_z_update", None)],
                                decision=dict(nb=_nb, side="U")))

# expansion slots per instance: B found at run time from trb_lin_expand_slots (shared W, GEMVs)
SLOT_CASES = [_case(f"slots{ns}_{lik}", N=120, M=80, B=None, prior=pr, lik=lik, shared=True, backend="gemv",
                    persist=-1, expect=[("k_z_update_chunked" if lik == "gaussian" else "k_z_update", None),
                                        ("k_x_update_chunked", None)]
                    + ([("k_reduce_slots", None)] if ns >= 5 else []),
                    absent=[] if ns >= 5 else ["k_reduce_slots"], decision=dict(ns=ns))
              for ns in (1, 2, 3, 4, 5) for pr, lik in (("gauss_bernoulli", "gaussian"), ("gaussian", "sgn"))]

# slots_of: B R G just below / just above 2^32, and the largest batch the sweep takes (several CTA
# boundaries inside instances whose row index times G exceeds 32 bits)
WORD_CASES = [_case(f"slots_word_{which}", N=512, M=512, B=which, shared=True, backend="gemv", persist=-1,
                    patterns=3, n_iter=6, expect=[("k_gemv_tma<1,2>", None), ("k_x_update_chunked", None)],
                    decision=dict(word=word))
              for which, word in (("below", "32-bit"), ("above", "64-bit"), ("max", "64-bit"))]

# chunks of 1024 elements in the x / z updates (Gaussian likelihood)
CHUNK_CASES = [_case(f"chunks_N{n}_M{m}", N=n, M=m, expect=[("k_x_update_chunked", -(-n // 1024)),
                                                            ("k_z_update_chunked", -(-m // 1024))])
               for n, m in ((1024, 1025), (1025, 1024), (2047, 3073), (3073, 2047))]

# cluster size of the one-CTA-per-instance updates: C doubles while n / (2C) >= 2048
CLUSTER_CASES = [
    _case("cluster_z_M16384_sgn", N=48, M=16384, prior="gaussian", lik="sgn", expect=[("k_z_update", 8)]),
    _case("cluster_z_M16384_abs", N=48, M=16384, prior="binary", lik="abs", n_iter=4, expect=[("k_z_update", 8)]),
    _case("cluster_z_M32768_sgn", N=64, M=32768, prior="gaussian", lik="sgn", expect=[("k_z_update", 16)]),
    _case("cluster_x_N16384", N=16384, M=48, upd=0, expect=[("k_x_update", 8)]),
    _case("cluster_x_N32768", N=32768, M=64, upd=0, expect=[("k_x_update", 16)]),
]

# persistent kernel: auto (-1), the cooperative grid (2), the 16-CTA cluster (3); shared memory
# 8 (2 ldmax + R) bytes against the 200 KB cap
_P = "k_sweep_persistent"
PERSIST_CASES = []
for _m, _n, _lik in ((1, 200, "gaussian"), (2, 201, "gaussian"), (15, 199, "sgn"), (16, 200, "gaussian")):
    for _mode in (-1, 2, 3):
        if _m < 16:
            exp = [(_P + "<false>", _m)] if _mode != 3 else []      # no cluster below 16 rows: fall back
            ab = [_P + "<.*>"] if _mode == 3 else []
        else:
            exp = [(_P + "<false>", 16)] if _mode == 2 else [(_P + "<true>", 16)]
            ab = []
        PERSIST_CASES.append(_case(f"persist_M{_m}_N{_n}_mode{_mode}", N=_n, M=_m, lik=_lik, persist=_mode,
                                   prior="gaussian" if _lik == "sgn" else "gauss_bernoulli",
                                   ref=f"persist_M{_m}_N{_n}", expect=exp, absent=ab))
for _mode in (-1, 2, 3):
    PERSIST_CASES.append(_case(f"persist_cap_N12768_mode{_mode}", N=12768, M=64, persist=_mode, n_iter=6,
                               ref="persist_cap_N12768",
                               expect=[(_P + ("<true>" if _mode == 3 else "<false>"), 16 if _mode == 3 else 64)]))
    PERSIST_CASES.append(_case(f"persist_over_N12784_mode{_mode}", N=12784, M=64, persist=_mode, n_iter=6,
                               ref="persist_over_N12784", expect=[("k_gemv_tma<16,2>", None)], absent=[_P + "<.*>"]))

# shared W with the default back end: stride-0 GEMVs below 16 instances, DMMA GEMMs from 16 on
SHARED_CASES = [
    _case("shared_B15", N=160, M=96, B=15, shared=True, persist=-1,
          expect=[("k_gemv_tma<1,2>", None)], absent=["k_dgemm_dmma(_tma)?"]),
    _case("shared_B16", N=160, M=96, B=16, shared=True, persist=-1,
          expect=[("k_dgemm_dmma(_tma)?", None), ("k_lin_rescale", None)], absent=["k_gemv_tma<.*"]),
]

# W shape and rank, schedules "general" and "auto" (damped: 3 passes, undamped: 2 passes)
SHAPE_CASES = []
for _name, _m, _n, _rd in (("tall", 150, 100, False), ("wide", 100, 150, False), ("square", 120, 120, False),
                           ("rankdef", 90, 130, True)):
    for _sched, _damp in (("general", 0.3), ("auto", 0.3), ("auto", 0.0)):
        SHAPE_CASES.append(_case(f"shape_{_name}_{_sched}_d{_damp}", N=_n, M=_m, B=3, rankdef=_rd,
                                 schedule=_sched, damping=_damp, persist=-1, ref=f"shape_{_name}_d{_damp}",
                                 expect=[("k_gemv_tma<1,.>", None)],
                                 decision=dict(schedule={"general": 0, "auto": 1 if _damp else 2}[_sched])))

ALL_CASES = GEMV_CASES + SLOT_CASES + WORD_CASES + CHUNK_CASES + CLUSTER_CASES + PERSIST_CASES + SHARED_CASES \
    + SHAPE_CASES


# ---------------------------------------------------------------- problems and references
_PRIOR_KW = dict(gauss_bernoulli=dict(rho=0.2), gaussian={}, binary=dict(p_pos=0.6))
_LIK_KW = dict(gaussian=dict(var=0.02), sgn={}, abs={})


def _problem(case, B, seed):
    """W ([M, N] shared / single, or [B, M, N]), x [K, N], y [K, M] for K distinct problems."""
    rng = np.random.RandomState(seed)
    N, M = case["N"], case["M"]
    K = case["patterns"] or B
    nW = 1 if (case["shared"] or B == 1) else B
    W = rng.randn(nW, M, N) / np.sqrt(N)
    if case["rankdef"]:
        W[:, 1] = W[:, 0]
    pk = case["prior"]
    if pk == "gauss_bernoulli":
        x = rng.randn(K, N) * (rng.rand(K, N) < 0.2)
    elif pk == "binary":
        x = np.where(rng.rand(K, N) < 0.6, 1.0, -1.0)
    else:
        x = rng.randn(K, N)
    z = np.einsum("bmn,bn->bm", W if nW == K else np.broadcast_to(W[0], (K, M, N)), x)
    lk = case["lik"]
    y = dict(gaussian=lambda: z + np.sqrt(0.02) * rng.randn(K, M), sgn=lambda: np.where(z >= 0, 1.0, -1.0),
             abs=lambda: np.abs(z))[lk]()
    return W, x, y


_REFS = {}


def _reference(case, W, x, y):
    """Oracle run per distinct problem: r_x [K, N], r_z [K, M], v_x [K], v_z [K], mse [n_iter, K]."""
    key = case["ref"]
    if key in _REFS:
        return _REFS[key]
    K = x.shape[0]
    ops_ = [_ref_op(W[k if W.shape[0] > 1 else 0]) for k in range(W.shape[0])]
    out = dict(r_x=[], r_z=[], v_x=[], v_z=[], mse=[])
    with _dense_means(), np.errstate(all="ignore"):
        for k in range(K):
            op = ops_[k if len(ops_) > 1 else 0]
            ref = orc.ep_glm(dict(kind=case["prior"], **_PRIOR_KW[case["prior"]]), op.W,
                             dict(kind=case["lik"], y=y[k], **_LIK_KW[case["lik"]]), case["n_iter"],
                             damping=case["damping"] or None, x_true=x[k], op=op)
            assert ref["n_iter"] == case["n_iter"]
            for name in ("r_x", "r_z", "v_x", "v_z"):
                out[name].append(ref[name])
            out["mse"].append(ref["traj"]["mse_x"])
    res = {k: np.array(v) for k, v in out.items()}
    res["mse"] = res["mse"].T
    res["rank"] = ops_[0].rank
    _REFS[key] = res
    return res


# ---------------------------------------------------------------- device run
def _kernel_key(name):
    m = re.search(r"k_gemv_tma<(\d+), ?(\d+)>", name) or re.search(r"k_gemv_tmaILi(\d+)ELi(\d+)E", name)
    if m:
        return f"k_gemv_tma<{m[1]},{m[2]}>"
    m = re.search(r"k_sweep_persistent<(true|false)>", name) or re.search(r"k_sweep_persistentILb([01])E", name)
    if m:
        return "k_sweep_persistent<%s>" % {"1": "true", "0": "false"}.get(m[1], m[1])
    if name.startswith("_Z"):
        m = re.search(r"(\d+)(k_\w+)", name)
        return m[2][:int(m[1])] if m else name
    m = re.search(r"\b(k_\w+)", name)
    return m[1] if m else name


def _trace_kernels(prof, path):
    """(kernel key, grid.x) of every kernel in the profile."""
    prof.export_chrome_trace(path)
    with open(path) as f:
        events = json.load(f)["traceEvents"]
    out = []
    for ev in events:
        if str(ev.get("cat", "")).lower() != "kernel":
            continue
        grid = (ev.get("args") or {}).get("grid")
        out.append((_kernel_key(ev.get("name", "")), int(grid[0]) if grid else None))
    return out


def _batch_size(case, lib):
    """Decision-driven batch sizes (the SM count is the device's)."""
    from tramp_b200 import ops
    B = case["B"]
    if "ns" in case["decision"]:
        R = min(case["N"], case["M"])
        want = case["decision"]["ns"]
        sm = lib.trb_device_sm_count()
        for B in range(1, 2 * sm + 1):
            if ops.lin_expand_slots(B, R) == want:
                return B
        pytest.fail(f"no batch of <= {2 * sm} instances has {want} expansion slots at R = {R}")
    if isinstance(B, str):
        R = min(case["N"], case["M"])
        G = lib.trb_device_sm_count()
        below = (2**32 - 1) // (G * R)      # largest B with B R G <= 2^32 - 1 (32-bit slots_of)
        B = dict(below=below, above=below + 1, max=65535)[B]
        assert B <= 65535
        assert B * R // 8 >= G                # the expansion runs on G = SM-count CTAs
    return B


@pytest.fixture(scope="module")
def lib():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from tramp_b200 import _lib
    return _lib.load()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ALL_CASES)
def test_sweep_geometry_matches_oracle(case, lib, tmp_path):
    import torch
    from torch.profiler import profile, ProfilerActivity
    from tramp_b200.priors import get_prior
    from tramp_b200.likelihoods import get_likelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import ExpectationPropagation, TrackErrors
    B = _batch_size(case, lib)
    N, M, n_iter = case["N"], case["M"], case["n_iter"]
    W, xk, yk = _problem(case, B, seed=sum(map(ord, case["ref"])))
    ref = _reference(case, W, xk, yk)
    K = xk.shape[0]
    idx = np.arange(B) % K
    if B == 1:
        Wd, x, y, prior = W[0], xk[0], yk[0], get_prior(size=N, prior_type=case["prior"], **_PRIOR_KW[case["prior"]])
    else:
        Wd = W[0] if case["shared"] else W
        x, y = xk[idx], yk[idx]
        prior = get_prior(size=N, prior_type=case["prior"], batch=B, **_PRIOR_KW[case["prior"]])
    lin = LinearChannel(Wd)
    lik = get_likelihood(y=y, likelihood_type=case["lik"], **_LIK_KW[case["lik"]])
    model = (prior @ V("x") @ lin @ V("z") @ lik).to_model()
    lib.trb_set_persistent_sweep(case["persist"])
    lib.trb_set_fused_rescale(case["fused"])
    lib.trb_set_update_kernels(case["upd"])
    try:
        ep = ExpectationPropagation(model)
        ep.schedule = case["schedule"]
        if case["backend"]:
            ep.linear_backend = case["backend"]
        lin._setup()                              # the factorisation is not part of the trace
        track = TrackErrors({"x": x})
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            ep.iterate(max_iter=n_iter, callback=track, damping=case["damping"])
            torch.cuda.synchronize()
        kernels = _trace_kernels(prof, str(tmp_path / "trace.json"))
    finally:
        lib.trb_set_persistent_sweep(-1)
        lib.trb_set_fused_rescale(1)
        lib.trb_set_update_kernels(-1)
    assert ep.n_iter == n_iter
    if "schedule" in case["decision"]:
        assert ep.last_schedule == case["decision"]["schedule"]
    if case["rankdef"]:
        assert lin.rank == ref["rank"] < lin.R

    # ---- the path: expected kernels (and grid.x where it is the decision), absent kernels
    keys = {k for k, _ in kernels}
    for pat, gx in case["expect"]:
        hit = [g for k, g in kernels if re.fullmatch(pat, k)]
        assert hit, f"{pat} did not run; kernels: {sorted(keys)}"
        if gx is not None:
            assert gx in hit, f"{pat} ran with grid.x {sorted(set(hit))}, expected {gx}"
    for pat in case["absent"]:
        assert not [k for k in keys if re.fullmatch(pat, k)], f"{pat} ran; kernels: {sorted(keys)}"

    # ---- the numbers: 1e-9 against the reference, natural scales as in test_sweep_matches_reference
    got = ep.get_variables_data()
    rx, rz = np.asarray(got["x"]["r"]).reshape(B, N), np.asarray(got["z"]["r"]).reshape(B, M)
    vx, vz = np.asarray(got["x"]["v"]).reshape(B), np.asarray(got["z"]["v"]).reshape(B)
    mse = np.array([np.atleast_1d(np.asarray(e["mse"])) for e in track.errors]).reshape(n_iter, B)
    zk = np.einsum("kmn,kn->km", W if W.shape[0] == K else np.broadcast_to(W[0], (K, M, N)), xk)
    tau_x, tau_z = np.mean(xk**2, axis=1)[idx], np.mean(zk**2, axis=1)[idx]
    for name, a in (("r_x", rx), ("r_z", rz)):
        r = ref[name][idx]
        scale = np.abs(r).max(axis=1, keepdims=True)
        bad = np.abs(a - r) > 1e-9 * np.abs(r) + 1e-9 * scale
        assert not bad.any(), f"{name}: instances {np.unique(np.nonzero(bad)[0])[:10]} deviate, " \
                              f"max |d| / scale = {np.max(np.abs(a - r) / scale):.3e}"
    for name, a, tau in (("v_x", vx, tau_x), ("v_z", vz, tau_z)):
        r = ref[name][idx]
        bad = np.abs(a - r) > 1e-9 * np.abs(r) + 1e-9 * tau
        assert not bad.any(), f"{name}: instances {np.nonzero(bad)[0][:10]} deviate"
    r = ref["mse"][:, idx]
    bad = np.abs(mse - r) > 1e-9 * r + 2e-9 * np.sqrt(r * tau_x)
    assert not bad.any(), f"mse: (iteration, instance) {np.argwhere(bad)[:10].tolist()} deviate"

    # ---- what this row covered
    SEEN["kernels"] |= keys
    SEEN["clusters"] |= {g for k, g in kernels if k in ("k_z_update", "k_x_update") and g}
    if "ns" in case["decision"]:
        from tramp_b200 import ops
        SEEN["ns"].add(ops.lin_expand_slots(B, min(N, M)))
    if "word" in case["decision"]:
        SEEN["slots_word"].add(case["decision"]["word"])
    del ep, model, lin
    if B > 1000:
        torch.cuda.empty_cache()


@pytest.mark.gpu
def test_every_kernel_choice_was_compared(lib):
    """The rows above, together, ran every TMA GEMV instantiation, both persistent variants, every
    slot count the update kernels sum themselves (and one the sweep reduces first), every cluster
    size and both word sizes of the slot arithmetic -- each compared with the reference.  If a
    dispatch threshold moves, this fails instead of leaving a boundary uncovered."""
    if not SEEN["kernels"]:
        pytest.skip("the geometry rows did not run in this session")
    want = {f"k_gemv_tma<{nb},{mode}>" for nb in (1, 2, 4, 8, 16) for mode in (0, 1, 2)}
    want |= {"k_sweep_persistent<true>", "k_sweep_persistent<false>"}
    assert not want - SEEN["kernels"], sorted(want - SEEN["kernels"])
    assert SEEN["ns"] >= {1, 2, 3, 4, 5}, SEEN["ns"]
    assert SEEN["clusters"] >= {1, 2, 4, 8, 16}, SEEN["clusters"]
    assert SEEN["slots_word"] == {"32-bit", "64-bit"}, SEEN["slots_word"]
