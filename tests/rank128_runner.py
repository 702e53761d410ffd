"""Child process of tests/test_gpu_rank128.py: the run-time switches of libgca (GCA_*) are latched at first use, so every
switch setting gets its own interpreter.  Runs the oracle parity of the adapter forward + backward at r = 128 for the
named case and prints ONE JSON line with the kernel variant libgca reported for every phase."""
import ctypes
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

import torch  # noqa: E402

from gconv_adapter_b200 import _cabi  # noqa: E402
from gconv_adapter_b200.graphs.synthetic import make_graph  # noqa: E402
from test_gpu_adapter import _oracle_parity  # noqa: E402

CASES = {
    # name: (workload, scale, d, r, overrides)
    "arxiv_relu": ("arxiv", 1 / 16, 256, 128, {}),
    "arxiv_silu_noskip": ("arxiv", 1 / 16, 300, 128, {"non_linearity": "silu", "skip_connection": False}),
    "cora_relu": ("cora", 1.0, 64, 128, {}),           # the fused small-graph kernels unless GCA_DISABLE_SMALL=1
}
# cases run after other (d, r) shapes in the same process: "name": [(d, r), ...] run first, then the case's own shape
PRELUDE = {
    # r 64 / d 128 asks the fused kernels for the same shared memory as r 128 / d 64, at a different occupancy
    "cora_after_r64": ("cora_relu", [(128, 64)]),
}


def main():
    case = sys.argv[1]
    base, pre = PRELUDE.get(case, (case, []))
    name, scale, d, r, over = CASES[base]
    lib = _cabi.load()
    ei, n = make_graph(name, seed=0, scale=scale)
    for d0, r0 in pre:
        _oracle_parity(ei, n, d0, r0, seed=40, tag=f"{case} prelude d={d0} r={r0}", **over)
    lib.gca_profile_enable(1)
    _oracle_parity(ei, n, d, r, seed=41, tag=case, **over)      # raises on any parity failure
    torch.cuda.synchronize()
    buf = ctypes.create_string_buffer(1 << 16)
    lib.gca_profile_report(buf, len(buf))
    lib.gca_profile_enable(0)
    prof = json.loads(buf.value.decode())
    print(json.dumps({"ok": True, "case": case, "n": n, "variants": {k: v["variant"] for k, v in prof.items()}}))


if __name__ == "__main__":
    main()
