"""Every run-time switch of libgca is product code: each one is exercised against the CPU oracle, forward + backward,
relu and silu, on arxiv-shaped (r = 16) and products-shaped (r = 32) graphs - including GCA_SPLIT_MB=0, which forces the
split K3 (plain hop + expand-only tcgen05 kernel) that full-size products-shaped graphs take by default.  The switches are
latched at first use, hence one subprocess per setting (tests/switch_runner.py); the child reports which kernel variant
ran in every phase and the test asserts it is the one the switch names."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
GCA_VARS = ("GCA_DISABLE_TC", "GCA_DISABLE_STREAM", "GCA_DISABLE_TMA", "GCA_DISABLE_PDL", "GCA_SPLIT_MB", "GCA_DISABLE_BWD_FUSE",
            "GCA_DISABLE_SMALL")


def run_case(case: str, env_over: dict) -> dict:
    env = {k: v for k, v in os.environ.items() if k not in GCA_VARS}
    env.update(env_over)
    res = subprocess.run([sys.executable, os.path.join(HERE, "switch_runner.py"), case], env=env, capture_output=True,
                         text=True, timeout=900)
    assert res.returncode == 0, f"{case} under {env_over}:\n{res.stdout[-3000:]}\n{res.stderr[-6000:]}"
    return json.loads(res.stdout.strip().splitlines()[-1])


# switch setting -> {phase: variant} that must be reported (r = 16 case / r = 32 case where they differ)
SETTINGS = {
    "default": ({}, {"project_fwd": "stream_f16", "bwd_up": "stream_f16", "hop_expand_fwd": "tcgen05", "hop_plain_bwd": "",
                     "expand_wgrad_bwd": "stream_f16"}),
    "no_bwd_fuse": ({"GCA_DISABLE_BWD_FUSE": "1"}, {"project_fwd": "stream_f16", "bwd_up": "stream_f16", "wgrad_down": "stream_f16",
                                                    "hop_expand_fwd": "tcgen05", "hop_expand_bwd": "tcgen05"}),
    "split_k3": ({"GCA_SPLIT_MB": "0", "GCA_DISABLE_BWD_FUSE": "1"},
                 {"hop_plain_fwd": "", "expand_fwd": "tcgen05", "hop_plain_bwd": "", "expand_bwd": "tcgen05"}),
    "no_stream": ({"GCA_DISABLE_STREAM": "1"}, {"project_fwd": "mma", "project_bwd": "mma", "wgrad_up": "mma", "wgrad_down": "mma",
                                                "hop_expand_fwd": "tcgen05"}),
    "no_tma": ({"GCA_DISABLE_TMA": "1"}, {"project_fwd": "mma", "wgrad_up": "mma", "hop_expand_fwd": "mma", "hop_expand_bwd": "mma"}),
    "no_tc": ({"GCA_DISABLE_TC": "1"}, {"project_fwd": "ffma", "project_bwd": "ffma", "wgrad_up": "ffma", "wgrad_down": "ffma",
                                        "hop_expand_fwd": "ffma", "hop_expand_bwd": "ffma"}),
    "no_pdl": ({"GCA_DISABLE_PDL": "1"}, {"project_fwd": "stream_f16", "hop_expand_fwd": "tcgen05"}),
}


@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("case", ["arxiv_relu", "arxiv_silu"])
def test_switch_parity_rank16(setting, case):
    env, expect = SETTINGS[setting]
    out = run_case(case, env)
    assert out["ok"]
    for phase, variant in expect.items():
        assert out["variants"].get(phase) == variant, f"{setting}: {phase} ran as {out['variants'].get(phase)!r}, all: {out['variants']}"


@pytest.mark.parametrize("setting", list(SETTINGS))
@pytest.mark.parametrize("case", ["products64_relu", "products64_silu_noskip"])
def test_switch_parity_rank32(setting, case):
    """r = 32: projection + weight gradient of the backward are two streaming launches (project_bwd, wgrad_up); with the
    streaming family off the projection runs on the tcgen05 / TMEM kernel."""
    env, expect = SETTINGS[setting]
    expect = dict(expect)
    if "bwd_up" in expect:
        v = expect.pop("bwd_up")
        expect["project_bwd"] = v
        expect["wgrad_up"] = v
    if "expand_wgrad_bwd" in expect:                        # the one-pass backward tail is an r = 16 kernel
        expect.pop("expand_wgrad_bwd")
        expect.pop("hop_plain_bwd")
        expect["hop_expand_bwd"] = "tcgen05"
        expect["wgrad_down"] = "stream_f16"
    if setting in ("no_stream", "no_tma"):
        expect["project_fwd"] = "tcgen05"
        expect.pop("project_bwd", None)
    out = run_case(case, env)
    assert out["ok"]
    for phase, variant in expect.items():
        assert out["variants"].get(phase) == variant, f"{setting}: {phase} ran as {out['variants'].get(phase)!r}, all: {out['variants']}"


SMALL_CASES = ["cora_relu", "cora_silu_noskip", "molecules_relu", "small_r32_noscalar", "small_r64_unnormalized", "small_powerlaw"]


@pytest.mark.parametrize("case", SMALL_CASES)
def test_small_graph_fused_path(case):
    """cora / molecule-batch sized graphs (n <= 4096) run the whole forward and the whole backward as ONE cooperative
    kernel each (gca_small.cu): parity against the oracle, and nothing else was launched."""
    out = run_case(case, {})
    assert out["ok"]
    assert out["variants"] == {"small_fwd": "fused", "small_bwd": "fused"}, out["variants"]
    if case == "small_powerlaw":
        assert out["max_in_degree"] > 512, out["max_in_degree"]      # the case really has hub rows


@pytest.mark.parametrize("case", SMALL_CASES)
def test_small_graph_through_the_phase_kernels(case):
    """GCA_DISABLE_SMALL=1: the same graphs through the per-phase kernels (the path they took before the fused one)."""
    out = run_case(case, {"GCA_DISABLE_SMALL": "1"})
    assert out["ok"]
    assert "small_fwd" not in out["variants"] and "small_bwd" not in out["variants"], out["variants"]
    assert "finalize" in out["variants"]
