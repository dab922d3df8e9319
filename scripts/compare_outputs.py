"""Compares two `bench.py --dump-outputs` directories written on the same seeded inputs by two builds.

    python scripts/compare_outputs.py REF_DIR NEW_DIR [--config S1|C3|C4|C5] [--tol 1e-5]

Every array is compared with max|a - b| <= tol · max|ref|; `grad_params` is split per parameter in `module.parameters()` order
(the layer for S1, PointConvResNet for C3-C5), so a small parameter is not judged against the scale of a large one.  A parameter
whose reference gradient is rounding noise (zero in exact arithmetic, e.g. the bias of a BatchNorm that feeds another
batch-statistics BatchNorm) is reported as such: its max|ref| is below 1e-4 of the largest gradient max of the step.
Exit status 1 if any other array exceeds the tolerance."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def param_shapes(config):
    """(name, numel) of every parameter in module.parameters() order, from a CPU instance of the benchmarked module."""
    import bench
    from crfconv_b200.continuous_crf_conv_big import ContinuousGaussianCRFConv
    from crfconv_b200.point_conv_big import PointConvResNet
    if config == "S1":
        m = ContinuousGaussianCRFConv(bench.CU, bench.CP, bench.CP, steps=1)
    else:
        m = PointConvResNet(6, bench.NET_CONFIGS[config]["classes"])
    return [(n, p.numel()) for n, p in m.named_parameters()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("ref")
    ap.add_argument("new")
    ap.add_argument("--config", default="S1")
    ap.add_argument("--tol", type=float, default=1e-5)
    args = ap.parse_args()
    names = sorted(f[:-4] for f in os.listdir(args.ref) if f.endswith(".npy"))
    assert names == sorted(f[:-4] for f in os.listdir(args.new) if f.endswith(".npy")), "the two dumps hold different arrays"
    rows = []
    for name in names:
        a, b = np.load(os.path.join(args.ref, name + ".npy")), np.load(os.path.join(args.new, name + ".npy"))
        assert a.shape == b.shape, f"{name}: shapes {a.shape} vs {b.shape}"
        if name == "grad_params":
            off = 0
            for pname, n in param_shapes(args.config):
                rows.append((f"grad_params[{pname}]", a[off:off + n], b[off:off + n]))
                off += n
            assert off == a.size, f"grad_params: {a.size} floats, parameters hold {off}"
        else:
            rows.append((name, a, b))
    gmax = max(float(np.abs(a).max()) for n, a, _ in rows if n.startswith("grad_params[")) if any(n.startswith("grad_params[") for n, _, _ in rows) else 0.0
    bad = 0
    print(f"{'array':60s} {'max|ref|':>11s} {'max|a-b|':>11s} {'rel':>10s}")
    for name, a, b in rows:
        ref = float(np.abs(a).max()) if a.size else 0.0
        diff = float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max()) if a.size else 0.0
        r = diff / ref if ref > 0 else (0.0 if diff == 0 else float("inf"))
        noise = name.startswith("grad_params[") and ref < 1e-4 * gmax
        ok = diff <= args.tol * ref or noise
        bad += not ok
        print(f"{name:60s} {ref:11.4e} {diff:11.4e} {r:10.2e}  {'ok' if ok and not noise else ('rounding noise' if noise else 'FAIL')}")
    print(f"{len(rows)} arrays, {bad} over {args.tol:g} x max|ref|")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
