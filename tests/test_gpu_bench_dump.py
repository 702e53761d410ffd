"""bench.py --dump-outputs: after the timed steps the benchmark writes what its last step computed (Y, gX and the parameter
gradients) as float32 .npy files within 64 MB; the inputs are seeded, so two runs with different --steps write the same
numbers, and Y is the oracle's."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from gconv_adapter_b200.graphs.synthetic import make_graph, make_inputs
from oracle.pyg_restated import GConvAdapterRef

from util import assert_close, load_module_params

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = {"y", "grad_x", "grad_scalar", "grad_conv_down.bias", "grad_conv_down.lin.weight", "grad_conv_up.bias",
         "grad_conv_up.lin.weight"}


def _bench(out_dir, steps):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cora", "--steps", str(steps),
                          "--warmup", "1", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    line = json.loads([ln for ln in res.stdout.splitlines() if ln.startswith("{")][-1])
    assert line["steps"] == steps
    return {f[:-4]: np.load(os.path.join(out_dir, f)) for f in os.listdir(out_dir)}


def test_dump_outputs_are_the_last_step_of_seeded_inputs(tmp_path):
    a = _bench(tmp_path / "a", 2)
    b = _bench(tmp_path / "b", 5)
    assert set(a) == set(b) == NAMES
    assert all(v.dtype == np.float32 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    for k in NAMES:
        assert_close(b[k], a[k], k)
    ei, n = make_graph("cora", seed=0)
    x, g_out, params = make_inputs(n, 64, 8, seed=0)
    assert a["y"].shape == a["grad_x"].shape == (n, 64)
    m = GConvAdapterRef(64, 8, learnable_scalar=True)
    load_module_params(m, params)
    with torch.no_grad():
        assert_close(a["y"], m(x, ei), "y")
