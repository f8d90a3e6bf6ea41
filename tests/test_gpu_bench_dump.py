"""GPU: bench.py --dump-outputs writes a fixed sample of every call's output of the last timed step, the same on every run
with the same arguments (what comparing two builds output for output relies on)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ARGS = ["--steps", "2", "--warmup", "1", "--no-e2e", "--no-cpu", "--no-generation", "--no-search", "--no-lowbit",
        "--no-reference-legs", "--no-other-configs"]


def test_dump_outputs_sample_every_call_and_repeat(tmp_path):
    from fpqvar_b200.var_workload import WORKLOADS
    hot = WORKLOADS["var_d30_w4a4_rot"]
    dumps = []
    for run in ("a", "b"):
        d = tmp_path / run
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *ARGS, "--dump-outputs", str(d)],
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
        line = json.loads(out.stdout.strip().splitlines()[-1])
        assert line["config"]["workload"] == hot.name and line["steps"] == 2
        dumps.append({f: np.load(d / f) for f in sorted(os.listdir(d))})
    a, b = dumps
    assert set(a) == {f"s{c.stage}_{c.site}.npy" for c in hot.calls()}
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    for f, v in a.items():
        assert v.dtype == np.float32 and v.ndim == 2 and v.shape[0] == hot.depth, f
        assert np.isfinite(v).all() and np.any(v != 0), f
        assert np.array_equal(v, b[f]), f

    # a dumped row is that call's output: recompute the first (re-launched) and the last (left in the arena) proj and fc2
    # calls from the same synthetic inputs, at the same seeded sample indices
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from fpqvar_b200.hotpath import run_call
    dev = torch.device("cuda", 0)
    arenas, _, _, plan = bench.synthetic_step(torch, hot, dev, 0)
    n = a["s0_proj.npy"].shape[1]
    for site in ("proj", "fc2"):
        ids = [i for i, (c, _, _) in enumerate(plan) if c.site == site]
        assert not bench.slice_intact(plan, ids[0]) and bench.slice_intact(plan, ids[-1])
        for i in (ids[0], ids[-1]):
            c, pi, _ = plan[i]
            src = bench.in_arena(arenas, c)
            off = (pi - src.base) // src.t.element_size()
            x = src.t[off:off + c.elems].view(c.rows, c.cols)
            idx = torch.from_numpy(np.random.default_rng(i).integers(0, c.elems, n)).to(dev)
            want = run_call(c, x).reshape(-1)[idx].float().cpu().numpy()
            assert np.array_equal(a[f"s{c.stage}_{c.site}.npy"][c.block], want), (site, i)
