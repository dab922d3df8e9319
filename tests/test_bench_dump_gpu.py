"""bench.py --dump-outputs end to end: the arrays of the last timed step are the same in every run, and the replayed CUDA graphs
hand back what the eager step computes on the same input set (3 timed steps rotate through 8 input sets: a dump of any other
set than the last one would not match)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests._util import rel_err_trimmed, rel_l2

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _dump(tmp_path, name, *extra):
    d = tmp_path / name
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--clouds", "1", "--steps", "3", "--warmup", "1",
                        "--pack-index", "off", "--dump-outputs", str(d), *extra], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    return {f[:-4]: np.load(d / f) for f in os.listdir(d)}


def test_dumped_outputs_repeat_and_match_the_eager_step(tmp_path):
    graph = _dump(tmp_path, "graph")
    assert sorted(graph) == ["grad_pairwise", "grad_params", "grad_unary", "grad_unary_rows", "out", "out_rows"]
    assert all(v.dtype == np.float32 for v in graph.values())
    assert graph["out"].shape == (32768, 64) and graph["grad_unary"].shape == (8192, 128)
    for name, other in (("graph_again", _dump(tmp_path, "graph_again")), ("eager", _dump(tmp_path, "eager", "--no-graph"))):
        assert sorted(other) == sorted(graph), name
        for k, a in graph.items():
            b = other[k]
            if k.endswith("_rows"):
                assert np.array_equal(a, b), (name, k)
            else:                           # floating-point atomics reorder sums: agreement to fp32 rounding, not bit for bit
                assert rel_err_trimmed(b, a) < 1e-4 and rel_l2(b, a) < 1e-5, (name, k, rel_err_trimmed(b, a), rel_l2(b, a))
