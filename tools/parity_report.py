"""Parity report: public API on the GPU vs the golden vectors of the reference.
Prints, per golden sweep and GEMV implementation, the max relative deviation of
every compared quantity.  Usage: python tools/parity_report.py"""
import json, os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
from tests.test_gpu_api import _build, _SeqInit, _configs
from tramp_b200.algos import ExpectationPropagation, TrackErrors, TrackEvolution, JoinCallback
from tests.golden import load_sweeps

sw = load_sweeps("tests/golden")
report = {}
for cfg in _configs(sw):
    name = cfg["name"]
    for impl in (1, 2):
        ep = ExpectationPropagation(_build(cfg, sw, name))
        ep.gemv_impl = impl
        track, evo = TrackErrors({"x": sw[name + "_x"]}), TrackEvolution()
        init = _SeqInit(sw, name) if cfg.get("init") == "noisy" else None
        ep.iterate(max_iter=cfg["n_iter"], callback=JoinCallback([track, evo]), initializer=init,
                   damping=cfg["damping"])
        mse = np.array([e["mse"] for e in track.errors]); df = evo.get_dataframe()
        d = ep.get_variables_data()
        rel = lambda a, b: float(np.max(np.abs(a - b) / np.maximum(np.abs(b), 1e-300)))
        relmax = lambda a, b: float(np.max(np.abs(a - b)) / (np.max(np.abs(b)) or 1.0))   # an all-zero reference: absolute
        x = sw[name + "_x"]
        r = dict(mse=rel(mse, sw[name + "_mse"]),
                 mse_cond=float(np.max(np.abs(mse - sw[name + "_mse"]) / (2 * np.sqrt(sw[name + "_mse"] * np.mean(x**2))))),
                 vx=rel(df[df.id == "x"].v.values, sw[name + "_vx"]),
                 vz=rel(df[df.id == "z"].v.values, sw[name + "_vz"]),
                 rx=relmax(d["x"]["r"], sw[name + "_rx"]), rz=relmax(d["z"]["r"], sw[name + "_rz"]))
        for k in range(1, 9):
            a, b = ep._edge(f"e{k}")
            r[f"e{k}_a"] = rel(np.asarray(a), sw[f"{name}_e{k}_a"])
            r[f"e{k}_b"] = relmax(b, sw[f"{name}_e{k}_b"])
        report[f"{name}/impl{impl}"] = r
        print(name, impl, {k: f"{v:.1e}" for k, v in r.items()}, flush=True)
# per golden: which quantities meet PLAIN 1e-9 relative (north star), which only the natural-scale
# tolerance of tests/test_gpu_api.py (cancellation in the reference's own formulas at a -> 1e6..AMAX)
summary = {}
for key, r in report.items():
    name = key.split("/")[0]
    sat = max(float(sw[f"{name}_e{k}_a"]) for k in range(1, 9)) > 1e4
    plain = {q: v <= 1e-9 for q, v in r.items() if q != "mse_cond"}
    summary[key] = dict(saturated_messages=bool(sat),
                        posterior_plain_1e9={q: plain[q] for q in ("mse", "vx", "vz", "rx", "rz")},
                        all_posterior_quantities_plain_1e9=all(plain[q] for q in ("mse", "vx", "vz", "rx", "rz")),
                        all_edges_plain_1e9=all(v for q, v in plain.items() if q.startswith("e")),
                        worst_edge=max((v, q) for q, v in r.items() if q.startswith("e"))[::-1],
                        mse_on_signal_scale=r["mse_cond"])
    print(key, summary[key], flush=True)
os.makedirs("gpurun_out", exist_ok=True)
json.dump(dict(max_rel_dev=report, summary=summary), open("gpurun_out/r02_parity_report.json", "w"), indent=1)
