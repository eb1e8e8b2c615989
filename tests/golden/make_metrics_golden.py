"""Generate tests/golden/metrics.npz from the UNMODIFIED reference functions
(openwakeword/metrics.py of the original openWakeWord project):
    python tests/golden/make_metrics_golden.py <openWakeWord checkout>
Series are built so that the reference does not raise (its grouping loop indexes one past a transition's 1, so a
series whose final element is a fresh 0->1 rise makes it throw IndexError)."""
import importlib.util
import os
import sys

import numpy as np


def load_reference_metrics(checkout):
    spec = importlib.util.spec_from_file_location("ref_metrics", os.path.join(checkout, "openwakeword", "metrics.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def series(rng, kind, T):
    if kind == 0:                                   # sparse spikes on a low floor
        s = rng.uniform(0, 0.05, T)
        idx = rng.integers(0, T, max(1, T // 40))
        s[idx] = rng.uniform(0.3, 1.0, idx.shape[0])
    elif kind == 1:                                 # dense alternation near the start (exercises the grouping rule)
        s = rng.uniform(0, 1, T)
    elif kind == 2:                                 # bursts of consecutive detections
        s = rng.uniform(0, 0.1, T)
        for p in rng.integers(0, max(1, T - 30), max(1, T // 60)):
            s[p:p + rng.integers(1, 25)] = rng.uniform(0.5, 1.0)
    else:                                           # smooth random walk through [0,1]
        s = np.clip(0.5 + np.cumsum(rng.normal(0, 0.08, T)), 0, 1)
    s[-1] = 0.0                                     # never end on a fresh rise (reference would raise IndexError)
    return s.astype(np.float32)


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    ref = load_reference_metrics(sys.argv[1])
    rng = np.random.default_rng(2024)
    out = {}
    lens = [7, 64, 500, 3000, 20000]
    sers, fps = [], []
    thr = np.linspace(0.01, 0.99, 25)
    windows = [1, 5, 50]
    for T in lens:
        for kind in range(4):
            s = series(rng, kind, T)
            sers.append(s)
            fps.append([[int(ref.get_false_positives(s, threshold=float(t), grouping_window=w)) for t in thr] for w in windows])
    out["n_series"] = np.int64(len(sers))
    for i, s in enumerate(sers):
        out[f"s{i}"] = s
    out["thresholds"] = thr
    out["windows"] = np.array(windows)
    out["fp"] = np.array(fps, dtype=np.int64)                       # [series][window][threshold]
    s = sers[14]
    out["roc_series"] = np.int64(14)
    out["roc_fprs"] = np.array(ref.generate_roc_curve_fprs(list(s), n_points=25, time_per_prediction=0.08, grouping_window=50))
    out["roc_tprs"] = np.array(ref.generate_roc_curve_tprs(s, n_points=25))
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "metrics.npz")
    np.savez_compressed(path, **out)
    print("wrote", path, "series", len(sers), "fp", out["fp"].shape, "nonzero grouping effect:",
          int((out["fp"][:, 0] != out["fp"][:, 2]).sum()))


if __name__ == "__main__":
    main()
