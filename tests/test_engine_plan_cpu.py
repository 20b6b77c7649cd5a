"""ResnetEngine's code-path plan (engine.resnet_plan), computed without weights or a device.

The shapes, channel counts, precisions and switches below are those of tests/test_engine_paths_gpu.py: together they must
reach every stem, every head and both forwards, so that a threshold change leaving a branch untested fails here."""
from deepliif_b200.engine import ResnetPlan, ResnetSwitches, resnet_plan
from test_engine_paths_gpu import PRECISIONS, RESNET_CASES, SWITCH_CASES, SWITCHES


def _plan(case, precision, switches=ResnetSwitches()):
    c = RESNET_CASES[case]
    return resnet_plan(c.H, c.W, (64, c.in_nc, 7, 7), (c.out_nc, 64, 7, 7), precision, "tc", switches)


def test_gpu_matrix_reaches_every_stem_head_and_forward():
    plans = {(case, p): _plan(case, p) for case in RESNET_CASES for p in PRECISIONS}
    for case in SWITCH_CASES:
        for name, value in SWITCHES:
            field = {"DLB_FUSED": "fused", "DLB_FUSE_RESIDUAL": "fuse_residual", "DLB_STEM_STREAM": "stem_stream",
                     "DLB_HEAD_STREAM": "head_stream", "DLB_FUSE_STEM": "fuse_stem", "DLB_FUSE_UP": "fuse_up",
                     "DLB_FUSE_HEAD": "fuse_head"}[name]
            plans[(case, name)] = _plan(case, "bf16x3", ResnetSwitches(**{field: value == "1"}))
    for k, p in plans.items():
        print(k, p)
    assert {p.fused for p in plans.values()} == {True, False}
    assert {p.stem for p in plans.values()} == {"stream", "tc_stem", "window"}
    assert {p.head for p in plans.values()} == {"stream", "tc"}
    # the rows the matrix names its cases after
    assert _plan("tall_narrow", "bf16x3").stem == "tc_stem" and _plan("very_tall", "bf16x3").stem == "tc_stem"
    assert _plan("tiny", "bf16x3") == ResnetPlan(True, "window", "tc")
    assert _plan("six_in", "bf16x3").stem == "window" and _plan("four_channel", "bf16x3").head == "tc"
    for case in ("odd66", "odd33x45", "w_only"):
        assert not _plan(case, "bf16x3").fused
    # fp16x3 turns both streaming kernels off
    assert all(p.stem != "stream" and p.head != "stream" for (case, prec), p in plans.items() if prec == "fp16x3")


def test_bench_shape_plans_the_streaming_fused_path():
    """The measured workload (512 x 512 tiles, bf16x3, default switches) runs the fused forward with both streaming
    kernels: a plan change that drops it onto another path shows here rather than as a slower benchmark."""
    p = resnet_plan(512, 512, (64, 3, 7, 7), (3, 64, 7, 7), "bf16x3", "tc", ResnetSwitches())
    assert p == ResnetPlan(True, "stream", "stream")


def test_switches_come_from_the_environment(monkeypatch):
    assert ResnetSwitches.from_env() == ResnetSwitches()
    monkeypatch.setenv("DLB_STEM_STREAM", "0")
    monkeypatch.setenv("DLB_FUSE_UP", "1")
    sw = ResnetSwitches.from_env(fused=False)
    assert sw == ResnetSwitches(fused=False, stem_stream=False, fuse_up=True)
    assert resnet_plan(512, 512, (64, 3, 7, 7), (3, 64, 7, 7)) == ResnetPlan(True, "tc_stem", "stream")


def test_direct_backend_and_odd_sizes_plan_the_layer_by_layer_forward():
    assert resnet_plan(64, 64, (64, 3, 7, 7), (3, 64, 7, 7), "bf16x3", "direct", ResnetSwitches()) == \
        ResnetPlan(False, "direct", "direct")
    assert resnet_plan(66, 64, (64, 3, 7, 7), (3, 64, 7, 7), "bf16x3", "tc", ResnetSwitches()) == \
        ResnetPlan(False, "window", "tc")
    # more than 8 input channels or more than 4 output channels: the fp32 direct kernels
    assert resnet_plan(64, 64, (64, 9, 7, 7), (5, 64, 7, 7), "bf16x3", "tc", ResnetSwitches()) == \
        ResnetPlan(False, "direct", "direct")
