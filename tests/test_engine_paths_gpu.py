"""Network-level parity of every ResnetEngine / UnetEngine code path with the float64 oracle.

ResnetEngine picks its forward (fused or layer by layer), its stem and its head from the input size, the channel counts,
the precision and the DLB_* switches (engine.resnet_plan); the trunk convs pick halo-strip or normalise-then-conv per
layer.  The cases below reach each of those branches (tests/test_engine_plan_cpu.py checks that on the CPU) and compare
the engine's fp32 output with oracle/nets.py evaluated in float64.  Every case asserts, in this order: the output shape,
the max-abs error, and that the case is informative (the output neither vanishes nor saturates the tanh).

Also here: the host-side descriptor checks of ops.py, and a TilePipeline whose networks change weights or precision
after a CUDA graph was captured."""
import math
import os
from collections import namedtuple

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import nets

pytestmark = pytest.mark.gpu

GATE = 1e-3                 # north-star parity gate (BASELINE.json), and the ceiling of every bound below
# asserted max-abs per precision group: 4x the largest value measured over this file's cases, capped at GATE.
# Measured on an NVIDIA B200 (1000 W power limit): bf16x3 4.8e-4 (4x = 1.9e-3, capped), fp16x3 8.4e-5.
BOUND = {"bf16x3": 1e-3, "fp16x3": 3.4e-4}
SWITCH_TOL = 1e-4           # one switch flipped vs the default path (the fused vs unfused bound of test_resnet_gpu.py)
COMPOSE_TOL = 1e-6          # a sample of an N-batch vs its own N=1 run (test_batched_tiles_equal_single_tile_results)
PRECISIONS = ("bf16x3", "fp16x3")

NORMS = ("batch", "instance", "none")
Case = namedtuple("Case", "N H W n_blocks in_nc out_nc paddings dropout norms", defaults=(NORMS,))
ZR = ("zero", "reflect")
RESNET_CASES = {
    # reflect pad 1 and per-sample statistics are undefined on the 1 x 1 trunk map (the reference raises there too)
    "tiny": Case(2, 4, 4, 1, 3, 3, ("zero",), False, ("none",)),  # window-pack stem, 1x1 trunk, non-streaming head
    "min8": Case(7, 8, 8, 2, 3, 3, ZR, True),                    # smallest streaming stem / head; CTA ranges span images
    "short_wide": Case(1, 8, 1024, 1, 3, 3, ZR, False),          # many stem / head column strips
    "tall_narrow": Case(2, 264, 16, 2, 3, 3, ZR, True),          # conv_tc_stem
    "very_tall": Case(1, 1032, 8, 1, 3, 3, ZR, False),           # conv_tc_stem, 258 x 2 trunk
    "ragged": Case(3, 36, 100, 2, 3, 3, ZR, True),               # ragged halo-strip trunk (9 x 25)
    "two_strip": Case(2, 68, 132, 3, 3, 3, ZR, False),           # head across two strips, fused residual, reflect border
    "nine": Case(2, 128, 128, 9, 3, 3, ZR, True),                # product-shaped trunk
    "no_blocks": Case(2, 32, 32, 0, 3, 3, ZR, False),            # down[1] feeds up[0] directly
    "one_channel": Case(2, 32, 48, 2, 1, 1, ZR, True),           # stem C=1, head CO=1
    "four_channel": Case(1, 32, 32, 2, 4, 4, ZR, False),         # stem C=4, head CO=4 (no streaming head)
    "six_in": Case(2, 32, 32, 2, 6, 3, ZR, True),                # C=6: window-pack stem at every size
    "odd66": Case(1, 66, 66, 2, 3, 3, ZR, False),                # layer-by-layer forward, ceil(h / 2) trunk
    "odd33x45": Case(2, 33, 45, 1, 3, 3, ZR, True),              # layer-by-layer forward, odd extents
    "w_only": Case(1, 64, 66, 1, 3, 3, ("zero",), False),        # layer-by-layer forward through W alone
}
SWITCH_CASES = ("min8", "tall_narrow", "two_strip")
# each flips one switch away from its default (engine.ResnetSwitches)
SWITCHES = (("DLB_FUSED", "0"), ("DLB_FUSE_RESIDUAL", "0"), ("DLB_STEM_STREAM", "0"), ("DLB_HEAD_STREAM", "0"),
            ("DLB_FUSE_STEM", "0"), ("DLB_FUSE_UP", "1"), ("DLB_FUSE_HEAD", "0"))
UNET_CASES = {"d5_32": (5, 3, 32, 32), "d5_32x64": (5, 2, 32, 64), "d7_128": (7, 2, 128, 128),
              "d7_128x256": (7, 2, 128, 256), "d5_96x160": (5, 2, 96, 160)}   # num_downs, N, H, W
MEASURED = {p: [] for p in PRECISIONS}


def _resnet_params():
    out = []
    for name, c in RESNET_CASES.items():
        for norm in c.norms:
            for pad in c.paddings:
                out.append((name, norm, pad))
    return out


# ---- weights and oracle ------------------------------------------------------------------------------------------------
def _fan_in_scaled(sd, transposed, gains):
    """norm='none': the N(0, 0.02) weights of make_state_dict shrink activations layer after layer until the output is a
    constant.  Rescale every conv weight to gain / sqrt(fan-in) so they stay O(1); a stride-2 ConvTranspose2d gathers
    about a quarter of its taps per output.  gains(key) -> gain."""
    out = dict(sd)
    for k, v in sd.items():
        if v.dim() != 4:
            continue
        fan = v.shape[0] * v.shape[2] * v.shape[3] / 4 if k in transposed else v.shape[1] * v.shape[2] * v.shape[3]
        out[k] = v / 0.02 * gains(k) / math.sqrt(fan)
    return out


def resnet_weights(name, norm, pad):
    c = RESNET_CASES[name]
    shapes = nets.resnet_param_shapes(c.in_nc, c.out_nc, 64, c.n_blocks, norm, c.dropout, pad)
    seed = 200 + list(RESNET_CASES).index(name) * 8 + NORMS.index(norm) * 2 + ZR.index(pad)
    sd = nets.make_state_dict(shapes, seed, "stress")
    if norm == "none":
        up = {f"model.{10 + c.n_blocks}.weight", f"model.{13 + c.n_blocks}.weight"}
        head = f"model.{17 + c.n_blocks}.weight"
        sd = _fan_in_scaled(sd, up, lambda k: 0.5 if ("conv_block" in k or k == head) else math.sqrt(2.0))
    return sd


def unet_weights(name, norm):
    nd = UNET_CASES[name][0]
    sd = nets.make_state_dict(nets.unet_param_shapes(nd, 64, 3, 3, norm), 300 + list(UNET_CASES).index(name) * 4
                              + NORMS.index(norm), "stress")
    if norm == "none":
        convt = {k for k in sd if k.endswith((".3.weight", ".5.weight"))}
        sd = _fan_in_scaled(sd, convt, lambda k: 0.5 if k == "model.model.3.weight" else math.sqrt(2.0))
    return sd


def _input(N, C, H, W, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand((N, C, H, W), generator=g) * 2 - 1


def _double(sd):
    return {k: (v if k.endswith("num_batches_tracked") else v.double()) for k, v in sd.items()}


def resnet_cfg(name, norm, pad):
    c = RESNET_CASES[name]
    return dict(n_blocks=c.n_blocks, norm=norm, use_dropout=c.dropout, padding_type=pad)


_ORACLE = {}


def resnet_case(name, norm, pad):
    """(x fp32, fp32 state_dict, float64 oracle output), cached per configuration and shape."""
    key = ("resnet", name, norm, pad)
    if key not in _ORACLE:
        c = RESNET_CASES[name]
        sd = resnet_weights(name, norm, pad)
        x = _input(c.N, c.in_nc, c.H, c.W, 17 + list(RESNET_CASES).index(name))
        with torch.no_grad():
            y = nets.resnet_forward(x.double(), _double(sd), norm_mode="sample", **resnet_cfg(name, norm, pad))
        _ORACLE[key] = (x, sd, y)
    return _ORACLE[key]


def unet_case(name, norm):
    key = ("unet", name, norm)
    if key not in _ORACLE:
        nd, N, H, W = UNET_CASES[name]
        sd = unet_weights(name, norm)
        x = _input(N, 3, H, W, 41 + list(UNET_CASES).index(name))
        with torch.no_grad():
            y = nets.unet_forward(x.double(), _double(sd), num_downs=nd, norm=norm, norm_mode="sample")
        _ORACLE[key] = (x, sd, y)
    return _ORACLE[key]


def resnet_block0_pre_relu(x, sd, *, n_blocks, norm, use_dropout, padding_type):
    """norm='none' ResnetGenerator with block 0's skip taken from down[1] BEFORE its ReLU: what the fused forward
    computed when a pending activation was not treated as needing materialisation.  float64, CPU."""
    assert norm == "none" and n_blocks > 0
    conv = lambda h, k, **kw: F.conv2d(h, sd[k + ".weight"], sd.get(k + ".bias"), **kw)
    h = F.relu(conv(nets._pad(x, 3, padding_type), "model.1"))
    h = F.relu(conv(h, "model.4", stride=2, padding=1))
    pre = conv(h, "model.7", stride=2, padding=1)
    h = F.relu(pre)
    c1, _, c2, _ = nets.resnet_block_conv_indices(padding_type, use_dropout)
    bp = 1 if padding_type != "zero" else 0
    idx = 10
    for b in range(n_blocks):
        p = f"model.{idx}.conv_block"
        t = F.relu(conv(nets._pad(h, bp, padding_type), f"{p}.{c1}", padding=1 - bp))
        t = conv(nets._pad(t, bp, padding_type), f"{p}.{c2}", padding=1 - bp)
        h = (pre if b == 0 else h) + t
        idx += 1
    for _ in range(2):
        h = F.relu(F.conv_transpose2d(h, sd[f"model.{idx}.weight"], sd.get(f"model.{idx}.bias"), stride=2, padding=1,
                                      output_padding=1))
        idx += 3
    idx += 1
    return torch.tanh(conv(nets._pad(h, 3, padding_type), f"model.{idx}"))


# ---- assertions ---------------------------------------------------------------------------------------------------------
def _check(label, y, ref, precision):
    """Shape, then max-abs against the bound of the precision group, then that the case can show an error."""
    y = y.cpu()
    assert tuple(y.shape) == tuple(ref.shape), f"{label}: output {tuple(y.shape)}, oracle {tuple(ref.shape)}"
    err = (y.double() - ref).abs().max().item()
    MEASURED[precision].append(err)
    std, sat = ref.std().item(), (ref.abs() > 0.98).double().mean().item()
    print(f"{label} {precision}: max|d| {err:.3e} (oracle std {std:.3f}, saturated {sat:.4f})")
    assert err <= BOUND[precision], f"{label} {precision}: max|d| {err:.3e}"
    assert std >= 0.05 and sat <= 0.05, f"{label}: uninformative oracle output (std {std:.3f}, saturated {sat:.4f})"
    return err


@pytest.fixture(scope="module")
def engine_mod():
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from deepliif_b200 import engine
    yield engine
    for p, errs in MEASURED.items():
        if errs:
            print(f"\nlargest max|d| over {len(errs)} {p} cases: {max(errs):.3e}")


def _resnet(engine_mod, name, norm, pad, precision, **kw):
    _, sd, _ = resnet_case(name, norm, pad)
    return engine_mod.ResnetEngine(sd, precision=precision, backend="tc", **resnet_cfg(name, norm, pad), **kw)


# ---- ResNet -------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("name,norm,pad", _resnet_params())
def test_resnet_path_matches_fp64_oracle(engine_mod, name, norm, pad, precision):
    x, sd, ref = resnet_case(name, norm, pad)
    eng = _resnet(engine_mod, name, norm, pad, precision)
    _check(f"resnet {name} {norm} {pad}", eng.forward(x.cuda()), ref, precision)


@pytest.mark.parametrize("name,pad", [(n, p) for n, c in RESNET_CASES.items() if c.n_blocks > 0 for p in c.paddings])
def test_norm_none_cases_can_see_a_pre_relu_block_skip(name, pad):
    """The norm='none' cases are sensitive to block 0 taking its skip operand before down[1]'s ReLU: that network
    differs from the oracle by at least 10x the gate (CPU only)."""
    x, sd, ref = resnet_case(name, "none", pad)
    with torch.no_grad():
        bad = resnet_block0_pre_relu(x.double(), _double(sd), **resnet_cfg(name, "none", pad))
    d = (bad - ref).abs().max().item()
    print(f"{name} {pad}: pre-ReLU skip vs oracle max|d| {d:.3e}")
    assert d >= 10 * GATE


@pytest.mark.parametrize("switch", SWITCHES, ids=[f"{k}={v}" for k, v in SWITCHES])
@pytest.mark.parametrize("pad", ZR)
@pytest.mark.parametrize("norm", ("batch", "none"))
@pytest.mark.parametrize("name", SWITCH_CASES)
def test_resnet_switch_matches_oracle_and_default_path(engine_mod, monkeypatch, name, norm, pad, switch):
    x, sd, ref = resnet_case(name, norm, pad)
    xd = x.cuda()
    y0 = _resnet(engine_mod, name, norm, pad, "bf16x3").forward(xd)
    monkeypatch.setenv(*switch)           # the switches are read when an engine is built
    eng = _resnet(engine_mod, name, norm, pad, "bf16x3")
    y1 = eng.forward(xd)
    _check(f"resnet {name} {norm} {pad} {switch[0]}={switch[1]}", y1, ref, "bf16x3")
    d = (y1 - y0).abs().max().item()
    print(f"  vs default path max|d| {d:.3e}")
    assert d <= SWITCH_TOL


@pytest.mark.parametrize("pad", ZR)
@pytest.mark.parametrize("name", SWITCH_CASES)
def test_resnet_batch_equals_single_sample_runs(engine_mod, name, pad):
    x, _, _ = resnet_case(name, "batch", pad)
    eng = _resnet(engine_mod, name, "batch", pad, "bf16x3")
    xd = x.cuda()
    yb = eng.forward(xd)
    for i in range(x.shape[0]):
        assert (yb[i:i + 1] - eng.forward(xd[i:i + 1])).abs().max().item() <= COMPOSE_TOL


# ---- UNet ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fused", ("", "0"), ids=("fused_default", "fused_off"))
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("norm", NORMS)
@pytest.mark.parametrize("name", list(UNET_CASES))
def test_unet_path_matches_fp64_oracle(engine_mod, monkeypatch, name, norm, precision, fused):
    monkeypatch.setenv("DLB_FUSED", fused)        # UnetEngine reads it at forward time; "" = default (on)
    nd = UNET_CASES[name][0]
    x, sd, ref = unet_case(name, norm)
    eng = engine_mod.UnetEngine(sd, num_downs=nd, norm=norm, precision=precision)
    xd = x.cuda()
    yb = eng.forward(xd)
    _check(f"unet {name} {norm} DLB_FUSED={fused or 'default'}", yb, ref, precision)
    for i in range(x.shape[0]):
        assert (yb[i:i + 1] - eng.forward(xd[i:i + 1])).abs().max().item() <= COMPOSE_TOL


# ---- descriptor checks --------------------------------------------------------------------------------------------------
def test_wrappers_refuse_tensors_that_disagree_with_the_descriptor(engine_mod):
    """Each wrapper gets one tensor whose extents differ from the descriptor's: it raises before the C call, so no
    kernel is launched."""
    import ctypes as C

    from deepliif_b200 import _lib, ops
    Err = _lib.DeepliifB200Error
    dev = "cuda"
    d = ops.conv_desc(2, 8, 8, [64], 64, 3, 3, 1, 1)
    w_hi, w_lo = ops.pack_weights_tc(d, torch.randn(64, 64, 3, 3, device=dev) * 0.02)
    good = torch.zeros((2, 8, 8, 64), dtype=torch.bfloat16, device=dev)
    bad = torch.zeros((2, 7, 8, 64), dtype=torch.bfloat16, device=dev)
    with pytest.raises(Err, match="conv_tc"):
        ops.conv_tc(d, [good], [bad], w_hi, w_lo)
    with pytest.raises(Err, match="conv_tc"):
        ops.conv_tc(d, [bad], [good], w_hi, w_lo)
    y = torch.zeros((2, 8, 8, 64), device=dev)
    with pytest.raises(Err, match="conv_tc_fused"):
        ops.conv_tc_fused(d, [dict(x=y, residual=torch.zeros((2, 8, 9, 64), device=dev))], w_hi, w_lo)
    with pytest.raises(Err, match="conv_tc_fused"):       # a border of 1: x must be the 6 x 6 interior
        ops.conv_tc_fused(d, [dict(x=y, border=1)], w_hi, w_lo)
    dd = ops.conv_desc(2, 8, 8, [3], 64, 7, 7, 1, 3)
    w_d = ops.pack_weights_direct(dd, torch.randn(64, 3, 7, 7, device=dev) * 0.02)
    with pytest.raises(Err, match="conv_direct"):
        ops.conv_direct(dd, torch.zeros((2, 8, 8, 3), device=dev), w_d, in_nchw=True)
    with pytest.raises(Err, match="conv_direct"):
        ops.conv_direct(dd, torch.zeros((2, 3, 8, 8), device=dev), w_d, in_nchw=False)
    sc = torch.ones((2, 64), device=dev)
    with pytest.raises(Err, match="norm_apply"):
        ops.norm_apply(y, torch.ones((1, 64), device=dev), sc)
    with pytest.raises(Err, match="norm_apply"):
        ops.norm_apply(y, sc, sc, residual=torch.zeros((2, 8, 8, 32), device=dev))
    # the C entry point itself refuses a null input (it returns before launching)
    out = torch.empty((2, 8, 8, 64), device=dev)
    rc = _lib.load().dlb_conv_direct_fwd(C.byref(dd), None, 1, None, None, 0, C.c_void_p(w_d.data_ptr()), None,
                                         C.c_void_p(out.data_ptr()), 0, 0, C.c_void_p(ops._raw_stream()))
    assert rc != 0
    torch.cuda.synchronize()


# ---- graph replay after a weight / precision change -----------------------------------------------------------------------
def _model_dir(root, seed0):
    from deepliif_b200.options import Options, print_options
    d = dict(model="DeepLIIF", name="m", checkpoints_dir=str(root), gpu_ids=(0,), input_nc=3, output_nc=3, ngf=64, ndf=64,
             net_g="resnet_2blocks", net_gs="unet_32", net_d="n_layers", norm="batch", no_dropout=False, padding="zero",
             init_type="normal", init_gain=0.02, modalities_no=4, seg_gen=True, input_no=1, scale_size=64, phase="train",
             modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"], seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25],
             loss_G_weights=[0.2] * 5, loss_D_weights=[0.2] * 5, mod_id_seg="S")
    print_options(Options(d_params=d, mode="train"), save=True)
    mdir = os.path.join(str(root), "m")
    g_shapes = nets.resnet_param_shapes(3, 3, 64, 2, "batch", True, "zero")
    s_shapes = nets.unet_param_shapes(5, 64, 3, 3, "batch")
    sds = {f"G{i}": nets.make_state_dict(g_shapes, seed0 + i, "stress") for i in range(1, 5)}
    sds.update({f"GS{i}": nets.make_state_dict(s_shapes, seed0 + 10 + i, "stress") for i in range(5)})
    for k, sd in sds.items():
        torch.save(sd, os.path.join(mdir, f"latest_net_{k}.pth"))
    return mdir


@pytest.mark.parametrize("change", ["weights", "precision"])
def test_graph_replay_follows_weight_and_precision_changes(engine_mod, tmp_path, monkeypatch, change):
    """A TilePipeline replays a captured CUDA graph without calling the networks.  After load_state_dict on the cached
    networks (or a new net.precision) the next run_batch must compute with the new weights (precision), exactly as a
    freshly loaded model directory does."""
    monkeypatch.delenv("DLB_NO_GRAPH", raising=False)
    from deepliif_b200.models import get_opt, init_nets, run_batch
    old_dir = _model_dir(tmp_path / "old", 70)
    new_dir = _model_dir(tmp_path / "new", 90) if change == "weights" else old_dir
    rng = np.random.default_rng(5)
    tiles = (rng.random((4, 64, 64, 3)) * 255).astype(np.uint8)
    init_nets.cache_clear()
    opt = get_opt(old_dir)
    nets_ = init_nets(old_dir, True, opt)
    first = run_batch(tiles, nets_, opt, opt.seg_weights)
    before = run_batch(tiles, nets_, opt, opt.seg_weights)          # captured and replayed
    for k in first:
        assert np.array_equal(first[k], before[k])
    for k, net in nets_.items():
        if change == "weights":
            own = net.state_dict()
            sd = torch.load(os.path.join(new_dir, f"latest_net_{k}.pth"), weights_only=True)
            net.load_state_dict({n: v for n, v in sd.items() if n in own})
        else:
            net.precision = "bf16"
    after = run_batch(tiles, nets_, opt, opt.seg_weights)
    init_nets.cache_clear()
    opt_new = get_opt(new_dir)
    fresh_nets = init_nets(new_dir, True, opt_new)
    if change == "precision":
        for net in fresh_nets.values():
            net.precision = "bf16"
    fresh = run_batch(tiles, fresh_nets, opt_new, opt_new.seg_weights)
    init_nets.cache_clear()
    assert set(after) == set(fresh)
    for k in after:
        assert np.array_equal(after[k], fresh[k]), f"{k}: the replay after the {change} change differs from a fresh model"
    changed = np.mean([np.mean(after[k] != before[k]) for k in after])
    print(f"{change}: {changed:.3f} of the output values changed")
    # sensitivity: new weights change most values (measured 0.99); single-pass bf16 operands move a good share of them by
    # at least one uint8 step (measured 0.36)
    assert changed > (0.5 if change == "weights" else 0.1)
