"""Benchmark of the EP-sweep hot path (metric and config from BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            # our arm (CUDA)
  python bench.py --impl reference --gpus N --steps K ...   # reference arm (CPU)
  python bench.py ... --dump-outputs DIR                    # + the last timed step's outputs as .npy

Workload ("config.workload"): batched teacher-student sparse GLM, BASELINE.json
configs[2]: GaussBernoulliPrior(N=4096, rho=0.1) @ LinearChannel(Gaussian W,
M=2048, alpha=0.5) @ GaussianLikelihood(var=1e-2), Bayes-optimal student,
ConstantInit(0, 0), no damping, fixed iteration count, 4096 instances over 8
GPUs = 512 independent instances per GPU (weak scaling; 4096 instances do not fit
one GPU: 412 GB of operators).  A "step" is one EP sweep of ITERS = 100 iterations
over the rank's 512 instances, general 4-pass schedule (16*R*(N+M) algorithmic
bytes per instance-iteration, SURVEY 8d).  Metric: instance-EP-iterations/s,
whole job.

 value : sweeps timed on the device (CUDA events), operators / observations
         resident in HBM, messages re-initialised on the device every step.
 e2e   : the same sweeps through the public API -- a new model from HOST (pinned)
         observations every step: H2D of y and x_true, ExpectationPropagation(...)
         .iterate(...), D2H of the posterior means/variances and the MSE records.
         Operator factors stay resident: `value` and `e2e` are SWEEP-ONLY rates.
 setup : the factorisation the reference does in LinearChannel.__init__ (and counts in its
         end-to-end time, examples/figures/benchmark.py:22), measured on REAL W =
         randn(M, N) / sqrt(N) for a sample of instances through `LinearChannel(W)`
         (hand-written block-Jacobi set-up), with `e2e_incl_setup` = the rate of the same
         sample with host W -> factorisation -> 100 iterations all counted, and the EP
         result of those instances checked against the oracle.  The other instances of
         the timed sweeps use exactly Gaussian W drawn directly in factored form
         (tramp_b200/synthetic.py) -- the sweep cost does not depend on how the factors
         were obtained.
 N > 1 : two more blocks, `row_sharded` (BASELINE configs[4]) and `shared_w` (configs[3]).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_DEFAULT, ALPHA, RHO, NOISE_VAR = 4096, 0.5, 0.1, 1e-2
INSTANCES_PER_GPU = 512
ITERS_PER_STEP = 100   # SURVEY 8(d): fixed 100 iterations per sweep
METRIC = "instance-EP-iterations/s, sparse GLM N=4096 alpha=0.5"
UNIT = "instance-iterations/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--instances", type=int, default=INSTANCES_PER_GPU, help="instances per GPU")
    ap.add_argument("--iters", type=int, default=ITERS_PER_STEP, help="EP iterations per step")
    ap.add_argument("--n", type=int, default=N_DEFAULT)
    ap.add_argument("--gemv-impl", type=int, default=0)
    ap.add_argument("--schedule", default="general", choices=["general", "gauss3", "gauss2", "auto"],
                    help="operator passes per iteration of the headline run (general = 4, SURVEY 8d)")
    ap.add_argument("--no-shortcut-modes", action="store_true",
                    help="skip the separately reported 3-pass / 2-pass Gaussian-likelihood schedules")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-instances", type=int, default=1)
    ap.add_argument("--setup-instances", type=int, default=16,
                    help="instances with real W factorised through LinearChannel(W) (0: skip the setup block)")
    ap.add_argument("--setup-parity-instances", type=int, default=8,
                    help="of those, how many are checked against the CPU oracle (rank 0)")
    ap.add_argument("--no-multi-gpu-blocks", action="store_true",
                    help="N > 1: skip the row_sharded / shared_w blocks")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed for rank 0's instances as DIR/<name>.npy "
                         "(float64, instances on axis 0): posterior means x_r [B, N], z_r [B, M], variances "
                         "x_v, z_v [B], records mse / vx / vz _per_iter [B, iters]; a fixed seeded sample of "
                         "the instances if the whole set exceeds 64 MB")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA arm (--impl ours)")
    return args


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = str(gpu_index)
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) >= 8 and f[0] == self.gpu:
                self.rows.append(f)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        clocks, reasons, smax, power = [], set(), None, []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for f in self.rows:
            try:
                clocks.append(float(f[1]))
                smax = float(f[2])
                power.append(float(f[3]))
            except ValueError:
                continue
            for nm, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        clocks.sort()
        med = clocks[len(clocks) // 2] if clocks else None
        return {"sm_mhz": med, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(clocks), "power_w_max": max(power) if power else None}


# --------------------------------------------------------------------------- CPU arm
def cpu_threads():
    try:
        from threadpoolctl import threadpool_info
        n = [p["num_threads"] for p in threadpool_info() if p.get("user_api") == "blas"]
        return max(n) if n else os.cpu_count()
    except Exception:
        return os.cpu_count()


def oracle_instance(np, N, M, seed):
    """One teacher-student instance drawn as the reference does
    (gaussian_ensemble.py:19-20, gauss_bernoulli_prior.py:38-42, gaussian_channel.py:12-15)."""
    rng = np.random.RandomState(seed)
    W = rng.randn(M, N) / np.sqrt(N)
    x = rng.standard_normal(N) * rng.binomial(n=1, size=N, p=RHO)
    y = W @ x + np.sqrt(NOISE_VAR) * rng.standard_normal(M)
    return W, x, y


def time_oracle(np, W, x, y, iters, steps, warmup):
    """The CPU restatement of the reference EP (oracle/, kind "port"): full SVD
    setup (timed separately), then `steps` sweeps of `iters` iterations."""
    from oracle import tramp_oracle as orc
    t0 = time.perf_counter()
    op = orc.LinearOp(W)                       # matrix_rank + full SVD (linear_channel.py:36-46)
    setup_s = time.perf_counter() - t0
    prior = dict(kind="gauss_bernoulli", rho=RHO)
    lik = dict(kind="gaussian", var=NOISE_VAR, y=y)
    for _ in range(warmup):
        orc.ep_glm(prior, W, lik, iters, x_true=x, op=op)
    times = []
    for _ in range(steps):
        t0 = time.perf_counter()
        out = orc.ep_glm(prior, W, lik, iters, x_true=x, op=op)
        times.append(time.perf_counter() - t0)
    return dict(setup_s=setup_s, step_s=times, out=out)


def _reference_worker(job):
    """One process of the instance-parallel mode: its own instance, one BLAS thread."""
    import numpy as np
    N, M, seed, iters, steps, warmup = job
    W, x, y = oracle_instance(np, N, M, seed)
    res = time_oracle(np, W, x, y, iters, steps, warmup)
    return dict(setup_s=res["setup_s"], step_s=res["step_s"])


def time_oracle_processes(N, M, iters, steps, warmup, procs):
    """Independent instances on all host cores: `procs` processes, one BLAS thread
    each (SURVEY 8d, CPU baseline mode ii).  Returns (instance-iterations/s, setup_s)."""
    import multiprocessing as mp
    saved = {k: os.environ.get(k) for k in ("OPENBLAS_NUM_THREADS", "OMP_NUM_THREADS", "MKL_NUM_THREADS")}
    for k in saved:
        os.environ[k] = "1"            # inherited by the spawned interpreters, before they import numpy
    try:
        ctx = mp.get_context("spawn")
        with ctx.Pool(procs) as pool:
            t0 = time.perf_counter()
            out = pool.map(_reference_worker, [(N, M, 5000 + p, iters, steps, warmup) for p in range(procs)])
            wall = time.perf_counter() - t0
    finally:
        for k, v in saved.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    # the processes start together and run the same work: the slowest one bounds the job
    slowest = max(sum(o["step_s"]) for o in out)
    return procs * iters * steps / slowest, max(o["setup_s"] for o in out), wall


REFERENCE_ITERS_PER_STEP = 25   # the reference arm's bounded step (every EP iteration costs the same)


def run_reference(args):
    """`--impl reference`: the reference's CPU path for the same metric/config, using all the
    host threads it can: (i) one instance at a time with every BLAS thread, and (ii) one instance
    per core, one BLAS thread each; the better of the two is the line's value.  Both modes time
    EXACTLY `--steps` steps after `--warmup` warm-up steps; a step is a bounded sample of the
    workload (REFERENCE_ITERS_PER_STEP iterations of one instance, or of one instance per core),
    so that the whole run ends within a few minutes.  The reference is pure Python (networkx < 2)
    and cannot travel to the GPU box, so the arm times the oracle port (oracle/tramp_oracle.py,
    pinned against the reference's golden vectors)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import numpy as np
    N = args.n
    M = int(ALPHA * N)
    it_step = min(args.iters, REFERENCE_ITERS_PER_STEP)
    W, x, y = oracle_instance(np, N, M, seed=1234)
    try:
        # torchrun exports OMP_NUM_THREADS=1 to its workers: give BLAS the whole host back
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count(), user_api="blas")
    except Exception:
        pass
    res = time_oracle(np, W, x, y, it_step, args.steps, args.warmup)
    total = sum(res["step_s"])
    value = it_step * args.steps / total
    setup_s = res["setup_s"]
    cores = cpu_threads()
    sample = (f"1 instance per step (N={N}, M={M}), {it_step} EP iterations per step, all BLAS threads; "
              f"matrix_rank + full SVD set-up {res['setup_s']:.1f} s excluded")
    modes = {"blas_threads": value}
    per_core = False
    procs = os.cpu_count() or 1
    if procs > 1:
        try:
            v_p, setup_p, _ = time_oracle_processes(N, M, it_step, args.steps, args.warmup, procs)
            modes["one_instance_per_core"] = v_p
            if v_p > value:
                value, cores, setup_s, per_core = v_p, procs, setup_p, True
                total = args.steps * procs * it_step / v_p           # the slowest process's timed steps
                sample = (f"{procs} instances per step, one process and one BLAS thread each (N={N}, M={M}), "
                          f"{it_step} EP iterations per step; matrix_rank + full SVD set-up {setup_p:.1f} s "
                          "per instance excluded")
        except Exception as e:                                      # report the threaded mode alone
            modes["one_instance_per_core_error"] = repr(e)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        # the workload is our arm's; `cpu_baseline.sample` says which bounded part of it a step timed
        "config": workload_config(N, M, args.instances, args.iters),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "setup_s_per_instance": setup_s, "modes_instance_iterations_per_s": modes,
        # the same arm with the factorisation counted (the reference's own end-to-end time includes it,
        # examples/figures/benchmark.py:22): one sweep of `ep_iterations_per_step` iterations per instance
        # (one instance per core: the SVDs of `procs` instances run side by side)
        "incl_setup": {"value": args.iters / (setup_s / (procs if per_core else 1) + args.iters / value),
                       "unit": UNIT, "note": "set-up SVD + 100-iteration sweep per instance, same mode as `value`"},
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 60 * 10**6      # data of --dump-outputs: with the .npy headers, under 64 MB


def dump_outputs(np, out_dir, arrays):
    """Write {name: array with instances on axis 0} as out_dir/<name>.npy in float64; when the set
    exceeds DUMP_LIMIT_BYTES, keep the same seeded sample of instances in every array."""
    B = len(next(iter(arrays.values())))
    total = sum(np.asarray(a, dtype=np.float64).nbytes for a in arrays.values())
    keep = np.arange(B)
    if total > DUMP_LIMIT_BYTES:
        keep = np.sort(np.random.RandomState(0).choice(B, max(1, B * DUMP_LIMIT_BYTES // total), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(np.asarray(a)[keep], dtype=np.float64))


def gemv_bytes_for_schedule(schedule, R, N, M):
    return {0: 16 * R * (N + M), 1: 8 * R * (2 * N + M), 2: 16 * R * N}[schedule]


def workload_config(N, M, instances_per_gpu, iters, schedule="general"):
    return {
        "workload": ("batched teacher-student sparse GLM (BASELINE.json configs[2]): "
                     f"GaussBernoulliPrior(N={N}, rho={RHO}) @ LinearChannel(Gaussian W, M={M}) @ "
                     f"GaussianLikelihood(var={NOISE_VAR}), ConstantInit(0,0), no damping, "
                     "SWEEP ONLY with the thin-SVD operators resident in HBM (factorisation: see `setup`), "
                     + {"general": "general 4-pass schedule", "gauss3": "3-pass Gaussian-likelihood schedule",
                        "gauss2": "2-pass Gaussian-likelihood schedule",
                        "auto": "cheapest exact schedule (2-pass)"}[schedule]),
        "N": N, "M": M, "alpha": ALPHA, "instances_per_gpu": instances_per_gpu,
        "ep_iterations_per_step": iters,
        "l2": ("inputs larger than L2 (operators of one rank: "
               f"{instances_per_gpu * 8 * min(M, N) * (N + M) / 1e9:.1f} GB >> 126 MB)"),
    }


# --------------------------------------------------------------------------- our arm
def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torch.distributed.run")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    from tramp_b200 import _lib, synthetic
    from tramp_b200.priors import GaussBernoulliPrior
    from tramp_b200.likelihoods import GaussianLikelihood
    from tramp_b200.channels import LinearChannel
    from tramp_b200.variables import SISOVariable as V
    from tramp_b200.algos import (ExpectationPropagation, TrackErrors, TrackEvolution, JoinCallback,
                                  ConstantInit)
    lib = _lib.load()

    N, B, iters = args.n, args.instances, args.iters
    M = int(ALPHA * N)
    R = min(M, N)
    # ---- setup (outside the timed region, reported as setup_s) ---------------
    t0 = time.perf_counter()
    data = synthetic.gaussian_glm_batch(B, N, M, RHO, NOISE_VAR, seed=1000 + rank,
                                        workers=min(16, os.cpu_count() or 8))
    torch.cuda.synchronize()
    setup_s = time.perf_counter() - t0
    linear = LinearChannel.from_factors(data["Ut"], data["s"], data["Vt"], Nx=M, Nz=N, rank=R)
    y_host = data["y"].cpu().pin_memory()
    x_host = data["x"].cpu().pin_memory()

    def new_ep(y, x_true):
        model = (GaussBernoulliPrior(size=N, rho=RHO, batch=B) @ V("x") @ linear @ V("z")
                 @ GaussianLikelihood(y=y, var=NOISE_VAR)).to_model()
        ep = ExpectationPropagation(model)
        ep.gemv_impl = args.gemv_impl
        ep.schedule = args.schedule
        return ep

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident timing: `value` --------------------------------------
    ep = new_ep(data["y"], data["x"])
    st = ep._ensure_state()
    st["x_true"] = ep._vec_to_dev(data["x"], "x")
    rec = {k: torch.zeros((iters, B), dtype=torch.float64, device="cuda") for k in ("mse", "vx", "vz")}
    ep.configure_damping(None)
    sw = ep._descriptor(rec, iters, None)
    init = ConstantInit(a=0, b=0)

    def device_step():
        ep.init_message_dag(init)          # device-side fills, no PCIe traffic
        st["active"].fill_(1)
        ep._run(sw, 0, iters, True)

    for _ in range(args.warmup):
        device_step()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    lib.trb_profile_reset(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        device_step()
    e1.record()
    barrier()
    dev_ms = e0.elapsed_time(e1)
    clocks = sampler.stop()
    gemv_ms = _lib.C.c_double(0.0)
    n_gemv = lib.trb_profile_gemv_ms(_lib.C.byref(gemv_ms))
    launches = int(lib.trb_profile_launches(-1))
    lib.trb_profile_reset(0)
    flags = st["flags"].cpu().numpy()
    assert not (flags & 3).any(), "NaN in EP messages during the benchmark"
    mse_final = float(rec["mse"][iters - 1].mean().item())
    if args.dump_outputs and rank == 0:
        # before the shortcut schedules below reuse the state
        got = ep.get_variables_data()
        dump_outputs(np, args.dump_outputs, {
            "x_r": got["x"]["r"], "x_v": got["x"]["v"], "z_r": got["z"]["r"], "z_v": got["z"]["v"],
            **{k + "_per_iter": rec[k].T.cpu().numpy() for k in ("mse", "vx", "vz")}})

    # ---- exact shortcut schedules for the Gaussian likelihood, reported separately
    # (SURVEY 8d honesty rule: bytes of the passes each schedule really streams)
    shortcut = {}
    if not args.no_shortcut_modes and args.schedule == "general":
        ref_mse = rec["mse"].clone()
        ref_rx, ref_vx = st["rx"].clone(), st["vx"].clone()
        steps_s = max(2, args.steps // 2)
        for mode, passes_bytes in (("gauss3", 8 * R * (2 * N + M)), ("gauss2", 16 * R * N)):
            ep.schedule = mode
            sw_m = ep._descriptor(rec, iters, None)

            def mode_step():
                ep.init_message_dag(init)
                st["active"].fill_(1)
                ep._run(sw_m, 0, iters, True)

            for _ in range(2):
                mode_step()
            barrier()
            lib.trb_profile_reset(1)
            m0, m1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            m0.record()
            for _ in range(steps_s):
                mode_step()
            m1.record()
            barrier()
            ms = m0.elapsed_time(m1)
            g_ms = _lib.C.c_double(0.0)
            n_g = lib.trb_profile_gemv_ms(_lib.C.byref(g_ms))
            lib.trb_profile_reset(0)
            dev = max(float(((st["rx"] - ref_rx).abs().max() / ref_rx.abs().max()).item()),
                      float(((st["vx"] - ref_vx).abs() / ref_vx).max().item()),
                      float(((rec["mse"] - ref_mse).abs() / ref_mse).max().item()))
            mm = torch.tensor([ms], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(mm, op=dist.ReduceOp.MAX)
            shortcut[mode] = {
                "value": world * B * iters * steps_s / (mm.item() / 1e3), "unit": UNIT, "steps": steps_s,
                "algorithmic_bytes_per_instance_iteration": passes_bytes,
                "operator_pass_launches": n_g,
                "achieved_gbs": passes_bytes * B * iters * steps_s / (g_ms.value / 1e3) / 1e9,
                "max_rel_dev_vs_general_schedule": dev,
            }
        ep.schedule = args.schedule
        rec["mse"].copy_(ref_mse)
        st["rx"].copy_(ref_rx)
        st["vx"].copy_(ref_vx)

    # ---- end-to-end timing through the public API: `e2e` ----------------------
    def e2e_step():
        y = y_host.to("cuda", non_blocking=True)
        xt = x_host.to("cuda", non_blocking=True)
        ep2 = new_ep(y, xt)
        track, evo = TrackErrors({"x": xt}), TrackEvolution(ids=["x"])
        ep2.iterate(max_iter=iters, callback=JoinCallback([track, evo]))
        out = ep2.get_variables_data(["x"])          # D2H of r_x [B, N] and v_x [B]
        return out, track

    for _ in range(args.warmup):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out, track = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    h2d = (y_host.numel() + x_host.numel()) * 8
    d2h = out["x"]["r"].nbytes + out["x"]["v"].nbytes + 5 * iters * B * 8 + 2 * B * 4

    # ---- max over ranks ---------------------------------------------------------
    tt = torch.tensor([dev_ms, e2e_s * 1e3, gemv_ms.value], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    dev_ms, e2e_ms, gemv_ms_max = tt.tolist()
    total_units = world * B * iters * args.steps
    value = total_units / (dev_ms / 1e3)
    e2e_value = total_units / (e2e_ms / 1e3)

    # ---- roofline of the dominant kernel (k_gemv_tma) --------------------------
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
    bytes_per_inst_iter = 16 * R * (N + M)           # SURVEY 8(d): four operator passes
    # this rank, all timed GEMV launches: 4 per iteration (ConstantInit b = 0 makes the
    # first-iteration U^T b6 a memset, so there is no fifth pass)
    gemv_bytes = bytes_per_inst_iter * B * iters * args.steps
    if args.schedule == "general":
        assert n_gemv == 4 * iters * args.steps, (n_gemv, iters, args.steps)
    else:   # the honesty rule: bytes of the passes this schedule streams
        bytes_per_inst_iter = gemv_bytes_for_schedule(ep.last_schedule, R, N, M)
        gemv_bytes = bytes_per_inst_iter * B * iters * args.steps
    achieved = gemv_bytes / (gemv_ms.value / 1e3) / 1e9
    traffic = None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum per launch from the committed ncu capture
        prof = json.load(open(os.path.join(ROOT, "profiles", "ncu_gemv_traffic.json")))
        if prof.get("instances_per_gpu") == B and prof.get("N") == N:
            traffic = prof["dram_bytes_per_launch_avg"]
    except Exception:
        pass
    roofline = {
        "bound": "hbm", "kernel": "k_gemv_tma (project / expand, cp.async.bulk ring)",
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
        "peak_source": peak_src, "traffic": traffic,
        "launches_timed": n_gemv, "avg_launch_ms": gemv_ms.value / max(n_gemv, 1),
        "algorithmic_bytes_per_launch": gemv_bytes / max(n_gemv, 1),
        "kernel_share_of_step": gemv_ms.value / dev_ms if world == 1 else gemv_ms_max / dev_ms,
    }

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(N, M, B, iters, args.schedule),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": launches,
        "roofline": roofline,
        "setup_s": setup_s,
        "final_mse_mean": mse_final,
        "hbm_roofline_inst_it_s_per_gpu": peak * 1e9 / bytes_per_inst_iter,
        "frac_of_hbm_roofline": value / world / (peak * 1e9 / bytes_per_inst_iter),
    }
    if shortcut:
        line["shortcut_schedules"] = shortcut

    # ---- set-up on real W (SURVEY 8d inputs), every rank its own sample -----------
    from tools import bench_blocks
    if args.setup_instances > 0:
        line["setup"] = bench_blocks.setup_block(
            N, M, args.setup_instances, iters, seed0=7000,
            parity_instances=(args.setup_parity_instances if world == 1 and not args.no_cpu_baseline else 0),
            rank=rank, world=world)
        line["e2e_incl_setup"] = line["setup"]["e2e_incl_setup"]
    line["setup_s_synthetic_factors"] = line.pop("setup_s")

    # ---- CPU baseline + full-size parity sample, rank 0 at N = 1 ---------------
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        nb = max(1, args.cpu_instances)
        steps_cpu, vals, dev_max, setup_cpu = 2, [], 0.0, 0.0
        got = ep.get_variables_data(["x"])
        for b in range(nb):
            W = synthetic.dense_W(data, b)
            x_b, y_b = data["x"][b].cpu().numpy(), data["y"][b].cpu().numpy()
            res = time_oracle(np, W, x_b, y_b, iters, steps_cpu, 1)
            vals.append(iters * steps_cpu / sum(res["step_s"]))
            setup_cpu += res["setup_s"]
            ref = res["out"]
            dev_max = max(dev_max, float(np.max(np.abs(got["x"]["r"][b] - ref["r_x"])) / np.max(np.abs(ref["r_x"]))),
                          float(abs(got["x"]["v"][b] - ref["v_x"]) / ref["v_x"]))
            mse_dev = rec["mse"][:, b].cpu().numpy()
            dev_max = max(dev_max, float(np.max(np.abs(mse_dev - np.array(ref["traj"]["mse_x"])) / np.array(ref["traj"]["mse_x"]))))
        line["cpu_baseline"] = {
            "value": float(np.mean(vals)), "unit": UNIT, "cores": cpu_threads(), "kind": "port",
            "sample": (f"instances 0..{nb - 1} of the GPU workload (same W, y), {iters} iterations x "
                       f"{steps_cpu} sweeps each after 1 warm-up sweep, one instance at a time with all "
                       f"BLAS threads; matrix_rank + full SVD setup {setup_cpu / nb:.1f} s/instance excluded"),
            "setup_s_per_instance": setup_cpu / nb,
        }
        line["parity_vs_oracle_full_size"] = {"instances": nb, "max_rel_dev_r_v_mse": dev_max, "tol": 1e-9}
    # ---- N > 1: the two other multi-GPU modes of SURVEY 8e --------------------------
    if world > 1 and not args.no_multi_gpu_blocks:
        del ep, st, sw, rec, data, linear
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        line["row_sharded"] = bench_blocks.row_sharded_block(rank=rank, world=world)
        line["shared_w"] = bench_blocks.shared_w_block(rank=rank, world=world)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
