"""Network executors: sequence the C-ABI kernels for the reference's generators / discriminators.

Each engine is built from a reference-format ``state_dict`` (same keys/shapes as the reference modules,
SURVEY.md §8b) and owns the repacked weights; ``forward`` enqueues only library kernels (see ops.py) on the
current CUDA stream.  Layer order follows

  ResnetGenerator         /root/reference/deepliif/models/networks.py:386-446 (+ ResnetBlock :479-513)
  UnetGenerator           networks.py:533-545 (+ UnetSkipConnectionBlock :573-615)
  NLayerDiscriminator     networks.py:636-660

Normalisation semantics: ``norm_mode='sample'`` = statistics per (n, c) — InstanceNorm2d, and also what the
reference's BatchNorm2d computes on its inference path (batch 1, running stats nulled,
deepliif/util/__init__.py:743-755), so batched tiles reproduce the reference's per-tile results;
``norm_mode='batch'`` = statistics pooled over the batch (training-mode BatchNorm2d).
"""
from dataclasses import dataclass

import torch

from . import ops
from .ops import (ACT_LRELU02, ACT_NONE, ACT_RELU, ACT_TANH, FMT_BF16, FMT_FP16, PAD_REFLECT, PAD_ZERO)


def _env_flag(name, default):
    import os
    v = os.environ.get(name)
    return default if v is None or v == "" else v not in ("0", "false", "False", "no")


# bench.py sets this to a list to collect (start_event, end_event, tiles) around every ResNet-block conv launch
# (roofline.achieved is measured live on the launching stream); None = no instrumentation.
BLOCK_CONV_EVENTS = None


def _block_conv(cv, acts, N, H, W, pad, fused=False):
    run = cv.run_fused if fused else cv.run_tc
    ev = BLOCK_CONV_EVENTS
    if ev is None:
        return run(acts, N, H, W, pad=pad)
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = run(acts, N, H, W, pad=pad)
    b.record()
    ev.append((a, b, N))
    return r


@dataclass
class Precision:
    """Operand format of the tensor-core convs.  split=True: hi/lo 16-bit planes, 3 MMAs per K step
    (fp32-grade products; parity default).  split=False: single pass (bf16/fp16 operand rounding)."""
    fmt: int = FMT_BF16
    split: bool = True

    @staticmethod
    def parse(name):
        table = {"bf16x3": Precision(FMT_BF16, True), "fp16x3": Precision(FMT_FP16, True),
                 "bf16": Precision(FMT_BF16, False), "fp16": Precision(FMT_FP16, False)}
        if name not in table:
            raise ValueError(f"precision [{name}] is not recognized (bf16x3 | fp16x3 | bf16 | fp16)")
        return table[name]


@dataclass
class Act:
    """An activation in HBM: fp32 NHWC and/or split 16-bit NHWC planes (optionally with a border)."""
    f32: torch.Tensor = None
    hi: torch.Tensor = None
    lo: torch.Tensor = None
    pad: int = 0


@dataclass
class Lazy:
    """An activation that is never written to HBM: the producer's raw fp32 conv output plus the normalisation
    (scale/shift), activation and residual add that the consuming convolution evaluates while it loads its operand
    (dlb_conv_tc_fwd_fused)."""
    x: torch.Tensor
    scale: torch.Tensor = None
    shift: torch.Tensor = None
    act: int = ACT_NONE
    residual: torch.Tensor = None

    def src(self, border=0, border_mode=PAD_ZERO, out=None):
        return dict(x=self.x, scale=self.scale, shift=self.shift, act=self.act, residual=self.residual, out=out,
                    border=border, border_mode=border_mode)


@dataclass(frozen=True)
class ResnetSwitches:
    """The DLB_* kernel-path switches of ResnetEngine, read from the environment when an engine is built."""
    fused: bool = True           # DLB_FUSED: fused-operand forward (norm + activation evaluated by the consuming conv)
    fuse_residual: bool = True   # DLB_FUSE_RESIDUAL: the next block's first conv also evaluates the skip add
    stem_stream: bool = True     # DLB_STEM_STREAM: row-streaming stem kernel (dlb_stem_conv_fwd)
    head_stream: bool = True     # DLB_HEAD_STREAM: row-streaming head kernel (dlb_head_conv_fwd)
    fuse_stem: bool = True       # DLB_FUSE_STEM: window operand built in shared memory (dlb_conv_tc_fwd_stem)
    # measured: 0.99 ms fused (TMA-staged) vs 0.67 ms apply + TMA conv for up1
    fuse_up: bool = False        # DLB_FUSE_UP: ConvTranspose convs read a fused operand
    fuse_head: bool = True       # DLB_FUSE_HEAD: the non-streaming head reads a fused operand

    @staticmethod
    def from_env(fused=None, fuse_residual=None):
        """fused / fuse_residual: explicit values override the environment."""
        return ResnetSwitches(
            fused=_env_flag("DLB_FUSED", True) if fused is None else bool(fused),
            fuse_residual=_env_flag("DLB_FUSE_RESIDUAL", True) if fuse_residual is None else bool(fuse_residual),
            stem_stream=_env_flag("DLB_STEM_STREAM", True), head_stream=_env_flag("DLB_HEAD_STREAM", True),
            fuse_stem=_env_flag("DLB_FUSE_STEM", True), fuse_up=_env_flag("DLB_FUSE_UP", False),
            fuse_head=_env_flag("DLB_FUSE_HEAD", True))


@dataclass(frozen=True)
class ResnetPlan:
    """Which ResnetEngine code path runs for one input size."""
    fused: bool   # True: _forward_fused; False: the layer-by-layer forward
    stem: str     # "stream" (stem_conv) | "tc_stem" (conv_tc_stem) | "window" (stem_window_pack + conv_tc) | "direct"
    head: str     # "stream" (head_conv) | "tc" (conv_tc[_fused] + head_finish) | "direct"


def _resnet_kernels(stem_shape, head_shape, prec, backend, sw):
    """Size-independent part of the plan: (stem_tc, stem_stream, head_tc, head_stream) for the stem / head weights
    (PyTorch Conv2d shapes (Cout, Cin, R, S))."""
    tc = backend == "tc"
    co, ci, R, S = stem_shape
    # stem on the tensor cores through the horizontal-window operand (K = 7 taps x 8 channel lanes = 64)
    stem_tc = tc and ci <= 8 and S <= 8 and co % 32 == 0
    # row-streaming stem kernel (dlb_stem_conv_fwd): C <= 4 -> 64, 7 x 7, split bf16
    stem_stream = (stem_tc and sw.stem_stream and co == 64 and ci <= 4 and R == 7 and S == 7
                   and prec.split and prec.fmt == FMT_BF16)
    co, ci, R, S = head_shape
    # head on the tensor cores with the horizontal taps moved into 32 virtual output channels (j = s*4 + co)
    head_tc = tc and co <= 4 and S <= 8 and ci % 64 == 0
    # row-streaming head kernel (dlb_head_conv_fwd): 64 -> co <= 3, 7 x 7, split bf16
    head_stream = (head_tc and sw.head_stream and ci == 64 and R == 7 and S == 7 and co <= 3
                   and prec.split and prec.fmt == FMT_BF16)
    return stem_tc, stem_stream, head_tc, head_stream


def resnet_plan(H, W, stem_shape, head_shape, precision="bf16x3", backend="tc", switches=None):
    """The forward, stem and head ResnetEngine runs for an [N, C, H, W] input.  stem_shape / head_shape: shapes of the
    generator's first and last Conv2d weights; switches: ResnetSwitches (default: read from the environment).  Needs no
    weights and no device.  The per-layer choice between halo-strip and normalise-then-conv stays with the layer."""
    prec = Precision.parse(precision) if isinstance(precision, str) else precision
    sw = ResnetSwitches.from_env() if switches is None else switches
    stem_tc, stem_stream, head_tc, head_stream = _resnet_kernels(stem_shape, head_shape, prec, backend, sw)
    if not (backend == "tc" and sw.fused and stem_tc and head_tc and H % 4 == 0 and W % 4 == 0):
        return ResnetPlan(False, "window" if stem_tc else "direct", "tc" if head_tc else "direct")
    if stem_stream and H >= 8 and W >= 8 and (W >= 32 or H <= 256):   # (one statistics slice per row tile must fit the workspace)
        stem = "stream"
    elif sw.fuse_stem and stem_shape[1] <= 4 and H >= 16 and W >= 8 and stem_shape[3] == 7:
        stem = "tc_stem"
    else:
        stem = "window"
    return ResnetPlan(True, stem, "stream" if head_stream and H >= 8 and W >= 8 else "tc")


def _tc_ok(cins, cout):
    return all(c % 64 == 0 for c in cins) and cout % 32 == 0


class ConvLayer:
    """One nn.Conv2d / nn.ConvTranspose2d with weights repacked for its kernel."""

    def __init__(self, weight, bias, *, transposed=False, stride=1, pad=0, output_padding=0, cins=None,
                 prec=Precision(), backend="tc", n_tile=0):
        self.transposed, self.stride, self.pad, self.output_padding = transposed, stride, pad, output_padding
        w = weight.detach().to(torch.float32).contiguous()
        if transposed:
            cin_total, self.cout, self.R, self.S = w.shape
        else:
            self.cout, cin_total, self.R, self.S = w.shape
        self.cins = list(cins) if cins is not None else [cin_total]
        assert sum(self.cins) == cin_total
        self.bias = bias.detach().to(torch.float32).contiguous() if bias is not None else None
        self.prec = prec
        self.n_tile = n_tile
        self.use_tc = backend == "tc" and _tc_ok(self.cins, self.cout)
        self.w_f32 = w          # kept for the data-gradient packing (training)
        d = ops.conv_desc(1, 8, 8, self.cins, self.cout, self.R, self.S, stride, pad, transposed, output_padding)
        self.w_packed = None
        if self.use_tc:
            self.w_hi, self.w_lo = ops.pack_weights_tc(d, w, prec.fmt, prec.split)
        else:
            assert len(self.cins) == 1, "direct kernel takes one source"
            self.w_packed = ops.pack_weights_direct(d, w)

    def desc(self, N, H, W, pad=None, pad_mode=PAD_ZERO):
        return ops.conv_desc(N, H, W, self.cins, self.cout, self.R, self.S, self.stride,
                             self.pad if pad is None else pad, self.transposed, self.output_padding, pad_mode)

    def run_tc(self, acts, N, H, W, pad=None, fuse_stats=True):
        """acts: list of Act (split planes).  H, W: extents of the (possibly border-padded) operand.
        Returns (y, stats_ws | None): with fuse_stats the epilogue leaves partial statistics in stats_ws."""
        d = self.desc(N, H, W, pad)
        oh, ow = ops.conv_out_shape(d)
        per_phase = (oh // self.stride) * (ow // self.stride) if self.transposed else oh * ow
        ws = ops.stats_workspace(N, oh * ow, self.cout, acts[0].hi.device) if (fuse_stats and per_phase >= 128) else None
        y = ops.conv_tc(d, [a.hi for a in acts], [a.lo for a in acts], self.w_hi, self.w_lo, self.bias,
                        self.prec.fmt, self.prec.split, self.n_tile, stats_ws=ws)
        return y, ws

    def run_fused(self, srcs, N, H, W, pad=None, fuse_stats=True):
        """Like run_tc, but the operand is evaluated in-kernel from `srcs` (list of Lazy.src() dicts, one per K-source).
        H, W: extents of the conv input including the sources' border."""
        d = self.desc(N, H, W, pad)
        oh, ow = ops.conv_out_shape(d)
        per_phase = (oh // self.stride) * (ow // self.stride) if self.transposed else oh * ow
        ws = ops.stats_workspace(N, oh * ow, self.cout, srcs[0]["x"].device) if (fuse_stats and per_phase >= 128) else None
        y = ops.conv_tc_fused(d, srcs, self.w_hi, self.w_lo, self.bias, self.prec.fmt, self.prec.split, self.n_tile,
                              stats_ws=ws)
        return y, ws

    # ---- training ------------------------------------------------------------------------------------------------
    def wgrad(self, x_act, dy_hi, dy_lo, N, H, W, pad=None):
        """dL/dW in the PyTorch weight layout from the forward operand planes and the output-gradient planes."""
        d = self.desc(N, H, W, pad)
        return ops.conv_wgrad(d, x_act.hi, x_act.lo, dy_hi, dy_lo, fmt=self.prec.fmt, split=self.prec.split)

    def dgrad(self, dy_hi, dy_lo, N, H, W, pad=None):
        """dL/dx (fp32 NHWC [N,H,W,Cin]) of the forward layer applied to an [N,H,W,Cin] input: the same weight
        tensor in the opposite role (Conv2d <-> ConvTranspose2d), so it runs on conv_tc."""
        assert len(self.cins) == 1
        pad = self.pad if pad is None else pad
        fd = self.desc(N, H, W, pad)
        oh, ow = ops.conv_out_shape(fd)
        if self.transposed:
            dd = ops.conv_desc(N, oh, ow, [self.cout], self.cins[0], self.R, self.S, self.stride, pad, False, 0)
        else:
            op = H - ((oh - 1) * self.stride - 2 * pad + self.R)
            dd = ops.conv_desc(N, oh, ow, [self.cout], self.cins[0], self.R, self.S, self.stride, pad, True, op)
        if getattr(self, "_wT", None) is None:
            self._wT = ops.pack_weights_tc(dd, self.w_f32, self.prec.fmt, self.prec.split)
        return ops.conv_tc(dd, [dy_hi], [dy_lo], self._wT[0], self._wT[1], None, self.prec.fmt, self.prec.split)

    def run_direct(self, x, N, H, W, *, pad_mode=PAD_ZERO, in_nchw=False, in_scale=None, in_shift=None,
                   in_act=ACT_NONE, out_act=ACT_NONE, out_nchw=False):
        d = self.desc(N, H, W, None, pad_mode)
        if self.w_packed is None:       # a tensor-core layer that meets a shape its kernel does not take: packed once
            assert len(self.cins) == 1, "direct kernel takes one source"
            self.w_packed = ops.pack_weights_direct(d, self.w_f32)
        return ops.conv_direct(d, x, self.w_packed, self.bias, in_nchw, in_scale, in_shift, in_act, out_act, out_nchw)


class _NormParams:
    def __init__(self, sd, key, norm, device):
        self.gamma = self.beta = None
        self.running = None            # (running_mean, running_var, num_batches_tracked, momentum) of a tracking BatchNorm2d
        if norm == "batch":
            self.gamma = sd[key + ".weight"].detach().to(device=device, dtype=torch.float32).contiguous()
            self.beta = sd[key + ".bias"].detach().to(device=device, dtype=torch.float32).contiguous()
            rm, rv, nbt = sd.get(key + ".running_mean"), sd.get(key + ".running_var"), sd.get(key + ".num_batches_tracked")
            # state_dict() hands out the module's own buffer storage: updating these in place IS updating the module
            if rm is not None and rv is not None and rm.is_cuda and rm.dtype == torch.float32 and rm.is_contiguous():
                self.running = (rm.detach(), rv.detach(), nbt.detach() if (nbt is not None and nbt.is_cuda) else None, 0.1)


# Optional device uint64 [1] mixed into every dropout seed (set by training.GraphedStep: a captured CUDA graph bakes the
# host-drawn seeds, the counter makes each replay draw new masks; forward and backward read the same value).
DROP_EPOCH = [None]


class _EngineBase:
    def __init__(self, norm, norm_mode, prec, backend, device):
        if norm not in ("batch", "instance", "none"):
            raise NotImplementedError("normalization layer [%s] is not found" % norm)
        self.norm, self.norm_mode, self.prec, self.backend, self.device = norm, norm_mode, prec, backend, device

    def _pooled(self):
        return self.norm == "batch" and self.norm_mode == "batch"

    def _stats(self, y, np_, ws=None, want_stats=False):
        """raw conv output -> (scale, shift[, mean, rstd]) or Nones for norm='none'.  ws: partial statistics already
        written by the conv epilogue (then y is not read again)."""
        if self.norm == "none" or np_ is None:
            return (None, None, None, None) if want_stats else (None, None)
        # training-mode BatchNorm2d (the train engines): the finalize kernel also moves the running statistics
        running = np_.running if getattr(self, "update_running_stats", False) else None
        if ws is not None:
            N, H, W, C = y.shape
            return ops.norm_finalize(ws, N, H * W, C, np_.gamma, np_.beta, self._pooled(), want_stats=want_stats,
                                     running=running)
        return ops.norm_stats(y, np_.gamma, np_.beta, self._pooled(), want_stats=want_stats, running=running)

    def _apply(self, y, scale, shift, act, *, residual=None, want_f32=False, want_split=True, pad=0,
               pad_mode=PAD_ZERO, drop=None):
        dp, dseed = drop if drop is not None else (0.0, 0)
        f32, hi, lo = ops.norm_apply(y, scale, shift, act, residual, want_f32, want_split, self.prec.fmt, pad,
                                     pad_mode, need_lo=self.prec.split, drop_p=dp, drop_seed=dseed,
                                     drop_epoch=DROP_EPOCH[0] if dp > 0 else None)
        return Act(f32, hi, lo, pad)

    def _conv(self, layer, act, N, H, W):
        """Run a conv on an Act with whichever kernel the layer was packed for.  Zero padding only."""
        if layer.use_tc:
            return layer.run_tc([act], N, H, W)
        return layer.run_direct(act.f32, N, H, W), None


class ResnetEngine(_EngineBase):
    """ResnetGenerator forward (eval semantics: dropout = identity)."""

    def __init__(self, sd, *, n_blocks=9, norm="batch", use_dropout=False, padding_type="zero", norm_mode="sample",
                 precision="bf16x3", backend="tc", device="cuda", n_tile=0, trunk_n_tile=0, fused=None, fuse_residual=None):
        prec = Precision.parse(precision) if isinstance(precision, str) else precision
        super().__init__(norm, norm_mode, prec, backend, device)
        # fused operand load (default on the tensor-core backend): norm + activation (+ skip add) are evaluated by the
        # consuming convolution; fuse_residual also folds the ResnetBlock skip add into the next block's first conv.
        # per-stage switches (measured choices, see DESIGN.md): the trunk always gains; the stem / head / ConvTranspose stages
        # have little MMA work per converted strip and are converter-bound
        self.switches = ResnetSwitches.from_env(fused, fuse_residual)
        if padding_type not in ("zero", "reflect"):
            raise NotImplementedError("padding [%s] is not implemented" % padding_type)
        self.n_blocks, self.padding_type = n_blocks, padding_type
        self.pad_mode = PAD_REFLECT if padding_type == "reflect" else PAD_ZERO
        g = lambda k: sd[k].to(device) if k in sd else None
        mk = lambda k, **kw: ConvLayer(g(k + ".weight"), g(k + ".bias"), prec=prec, backend=backend, n_tile=n_tile, **kw)
        nrm = lambda k: _NormParams(sd, k, norm, device)
        # stem: on the tensor cores through the horizontal-window operand (K = 7 taps x 8 channel lanes = 64),
        # else (validation backend / exotic channel counts) on the fp32 direct kernel.  head: direct kernel.
        w1 = g("model.1.weight")
        idx_head = 4 + 3 * 2 + n_blocks + 3 * 2 + 1
        wh, bh = g(f"model.{idx_head}.weight"), g(f"model.{idx_head}.bias")
        self.stem_shape, self.head_shape = tuple(w1.shape), tuple(wh.shape)
        self.stem_tc, self.stem_stream, self.head_tc, self.head_stream = _resnet_kernels(
            self.stem_shape, self.head_shape, prec, backend, self.switches)
        if self.stem_tc:
            co, ci, R, S = w1.shape
            wk = torch.zeros((co, 64, R, 1), dtype=torch.float32, device=device)
            # wk[co, s*8 + c, r, 0] = w[co, c, r, s]
            wk.view(co, 8, 8, R)[:, :S, :ci, :] = w1.to(torch.float32).permute(0, 3, 1, 2)
            self.stem = ConvLayer(wk, g("model.1.bias"), pad=0, prec=prec, backend="tc", n_tile=n_tile)
            self.stem_S, self.stem_in_nc = S, ci
            self.stem_wpk = ops.stem_conv_pack(w1) if self.stem_stream else None
        else:
            self.stem = ConvLayer(w1, g("model.1.bias"), pad=3, backend="direct")
        self.stem_norm = nrm("model.2")
        idx = 4
        self.down, self.down_norm = [], []
        for _ in range(2):
            self.down.append(mk(f"model.{idx}", stride=2, pad=1)); self.down_norm.append(nrm(f"model.{idx + 1}"))
            idx += 3
        padm = 0 if padding_type == "zero" else 1
        c1 = padm; n1 = c1 + 1; c2 = n1 + 2 + (1 if use_dropout else 0) + padm; n2 = c2 + 1
        self.blocks = []
        for _ in range(n_blocks):
            pre = f"model.{idx}.conv_block"
            mkb = lambda k: ConvLayer(g(k + ".weight"), g(k + ".bias"), prec=prec, backend=backend, pad=1,
                                      n_tile=trunk_n_tile or n_tile)
            self.blocks.append((mkb(f"{pre}.{c1}"), nrm(f"{pre}.{n1}"), mkb(f"{pre}.{c2}"), nrm(f"{pre}.{n2}")))
            idx += 1
        self.up, self.up_norm = [], []
        for _ in range(2):
            self.up.append(mk(f"model.{idx}", transposed=True, stride=2, pad=1, output_padding=1))
            self.up_norm.append(nrm(f"model.{idx + 1}"))
            idx += 3
        # head: on the tensor cores with the horizontal taps moved into 32 virtual output channels (j = s*4 + co),
        # followed by the shifted-sum finish; else the fp32 direct kernel.
        if self.head_tc:
            co, ci, R, S = wh.shape
            wv = torch.zeros((32, ci, R, 1), dtype=torch.float32, device=device)
            # wv[s*4 + co, c, r, 0] = w[co, c, r, s]
            wv.view(8, 4, ci, R)[:S, :co] = wh.to(torch.float32).permute(3, 0, 1, 2)
            self.head = ConvLayer(wv, None, pad=0, prec=prec, backend="tc", n_tile=32)
            self.head_bias = bh.detach().to(torch.float32).contiguous() if bh is not None else None
            self.head_S, self.head_co = S, co
            self.head_wpk = ops.head_conv_pack(wh) if self.head_stream else None
        else:
            self.head = ConvLayer(wh, bh, pad=3, backend="direct")

    @torch.no_grad()
    def forward(self, x, taps=None):
        """x: fp32 NCHW [N,3,H,W] CUDA -> fp32 NCHW [N,3,H,W]."""
        x = x.contiguous()
        N, _, H, W = x.shape
        plan = self.plan(H, W)
        if plan.fused:
            return self._forward_fused(x, plan, taps)
        tc = self.backend == "tc"
        refl = self.pad_mode == PAD_REFLECT
        want = dict(want_f32=not tc, want_split=tc)

        def tap(name, a):
            if taps is not None:
                taps[name] = a

        # stem: Pad3 + Conv7x7 (NCHW input read directly) -> norm -> ReLU
        if plan.stem == "window":
            xh, xl = ops.stem_window_pack(x, 3, self.stem_S, self.pad_mode, self.prec.fmt, self.prec.split)
            y, ws = self.stem.run_tc([Act(None, xh, xl)], N, H + 6, W)
        else:
            y, ws = self.stem.run_direct(x, N, H, W, pad_mode=self.pad_mode, in_nchw=True), None
        tap("stem_conv", y)
        sc, sh = self._stats(y, self.stem_norm, ws)
        a = self._apply(y, sc, sh, ACT_RELU, **want)
        h, w = H, W
        # two stride-2 down convs (an odd extent gives ceil(h / 2): the extents are taken from each conv's output)
        for i in range(2):
            if tc and (h % 2 or w % 2):
                # the tensor-core stride-2 conv takes even extents only: the fp32 direct kernel evaluates the previous
                # layer's norm + ReLU while it loads that layer's raw output
                y, ws = self.down[i].run_direct(y, N, h, w, in_scale=sc, in_shift=sh, in_act=ACT_RELU), None
            else:
                y, ws = self._conv(self.down[i], a, N, h, w)
            h, w = y.shape[1], y.shape[2]
            sc, sh = self._stats(y, self.down_norm[i], ws)
            last = i == 1
            # the trunk keeps an fp32 residual stream next to the operand planes
            a = self._apply(y, sc, sh, ACT_RELU, want_f32=(not tc) or last, want_split=tc,
                            pad=1 if (refl and last and tc and self.n_blocks > 0) else 0, pad_mode=self.pad_mode)
            tap(f"down{i}", a)
        # ResNet blocks: x + Norm(Conv(ReLU(Norm(Conv(x)))))
        for b, (cv1, nm1, cv2, nm2) in enumerate(self.blocks):
            last = b == self.n_blocks - 1
            if tc:
                p = 1 if refl else 0
                y, ws = _block_conv(cv1, [a], N, h + 2 * p, w + 2 * p, 0 if refl else 1)
                sc, sh = self._stats(y, nm1, ws)
                t = self._apply(y, sc, sh, ACT_RELU, pad=p, pad_mode=self.pad_mode)
                y, ws = _block_conv(cv2, [t], N, h + 2 * p, w + 2 * p, 0 if refl else 1)
                sc, sh = self._stats(y, nm2, ws)
                a = self._apply(y, sc, sh, ACT_NONE, residual=a.f32, want_f32=True,
                                pad=0 if last else p, pad_mode=self.pad_mode)
            else:
                y = cv1.run_direct(a.f32, N, h, w, pad_mode=self.pad_mode)
                sc, sh = self._stats(y, nm1)
                y = cv2.run_direct(y, N, h, w, pad_mode=self.pad_mode, in_scale=sc, in_shift=sh, in_act=ACT_RELU)
                sc, sh = self._stats(y, nm2)
                a = self._apply(y, sc, sh, ACT_NONE, residual=a.f32, want_f32=True, want_split=False)
            tap(f"block{b}", a)
        # two ConvTranspose upsamplings
        for i in range(2):
            y, ws = self._conv(self.up[i], a, N, h, w)
            h, w = y.shape[1], y.shape[2]
            sc, sh = self._stats(y, self.up_norm[i], ws)
            if i == 0:
                a = self._apply(y, sc, sh, ACT_RELU, **want)
                tap("up0", a)
        # head: (norm + ReLU fused into the load) Pad3 + Conv7x7 + bias + Tanh, NCHW out
        if plan.head == "tc":
            a = self._apply(y, sc, sh, ACT_RELU, pad=3, pad_mode=self.pad_mode)
            z, _ = self.head.run_tc([a], N, h + 6, w + 6, fuse_stats=False)
            return ops.head_finish(z, self.head_bias, w, self.head_S, self.head_co, ACT_TANH)
        return self.head.run_direct(y, N, h, w, pad_mode=self.pad_mode, in_scale=sc, in_shift=sh, in_act=ACT_RELU,
                                    out_act=ACT_TANH, out_nchw=True)

    def plan(self, H, W):
        """The forward / stem / head this engine runs for an [N, C, H, W] input (see resnet_plan)."""
        return resnet_plan(H, W, self.stem_shape, self.head_shape, self.prec, self.backend, self.switches)

    def _consume(self, layer, lazy, N, H, W, *, pad=None, border=0, keep=False, fuse_stats=True, block=False, allow=(2,)):
        """Run `layer` on the lazy activation.  Strip-eligible layers evaluate it in-kernel (no HBM pass); the others
        (stride 2, maps below 16 x 8) get their operand planes from one dlb_norm_apply pass.  keep: also materialise the
        evaluated activation in fp32 (the ResnetBlock residual stream).  Returns (y, stats_ws, kept fp32 | None)."""
        Hv, Wv = H + 2 * border, W + 2 * border
        d = layer.desc(N, Hv, Wv, pad)
        kept = None
        mode = ops.conv_tc_fused_mode(d, self.prec.split, layer.n_tile) if (allow and layer.use_tc) else 0
        # 4 / 1: efficient only when the kernel can stage the source by TMA — a plain source behind no or a zero border
        plain = lazy.residual is None and not keep and (border == 0 or self.pad_mode == PAD_ZERO)
        if mode in allow and (mode == 2 or plain):
            if keep:
                kept = torch.empty_like(lazy.x)
            srcs = [lazy.src(border, self.pad_mode, out=kept)]
            y, ws = (_block_conv(layer, srcs, N, Hv, Wv, pad, fused=True) if block
                     else layer.run_fused(srcs, N, Hv, Wv, pad, fuse_stats=fuse_stats))
            return y, ws, kept
        a = self._apply(lazy.x, lazy.scale, lazy.shift, lazy.act, residual=lazy.residual, want_f32=keep, pad=border,
                        pad_mode=self.pad_mode)
        y, ws = (_block_conv(layer, [a], N, Hv, Wv, pad) if block else layer.run_tc([a], N, Hv, Wv, pad, fuse_stats=fuse_stats))
        return y, ws, a.f32

    @torch.no_grad()
    def _forward_fused(self, x, plan, taps=None):
        """The same network with (almost) no normalise/split pass between convolutions: a strip-eligible conv reads its
        producer's raw fp32 output and evaluates norm + ReLU (+ the block's skip add, + the reflect / zero border) while
        loading; with fuse_residual the skip add of block b is evaluated by the first conv of block b+1, which also
        writes the fp32 residual stream out once."""
        N, _, H, W = x.shape
        refl = self.pad_mode == PAD_REFLECT
        b = 1 if refl else 0
        bpad = 0 if refl else 1

        def tap(name, a):
            if taps is not None:
                taps[name] = a

        if plan.stem == "stream":
            ws = ops.stats_workspace(N, H * W, self.stem.cout, x.device)
            y = ops.stem_conv(x, self.stem_wpk, self.stem.bias, self.stem.cout, self.pad_mode, stats_ws=ws)
        elif plan.stem == "tc_stem":
            ws = ops.stats_workspace(N, H * W, self.stem.cout, x.device)
            y = ops.conv_tc_stem(x, 3, self.stem_S, self.pad_mode, self.stem.cout, self.stem.w_hi, self.stem.w_lo, self.stem.bias,
                                 self.prec.fmt, self.prec.split, self.stem.n_tile, stats_ws=ws)
        else:
            xh, xl = ops.stem_window_pack(x, 3, self.stem_S, self.pad_mode, self.prec.fmt, self.prec.split)
            y, ws = self.stem.run_tc([Act(None, xh, xl)], N, H + 6, W)
        tap("stem_conv", y)
        sc, sh = self._stats(y, self.stem_norm, ws)
        cur = Lazy(y, sc, sh, ACT_RELU)
        h, w = H, W
        for i in range(2):
            y, ws, _ = self._consume(self.down[i], cur, N, h, w)
            h, w = h // 2, w // 2
            sc, sh = self._stats(y, self.down_norm[i], ws)
            cur = Lazy(y, sc, sh, ACT_RELU)
        for bi, (cv1, nm1, cv2, nm2) in enumerate(self.blocks):
            # the block input is also its skip operand: unless cur.x already holds it (no pending norm, activation or
            # skip add), it is materialised in fp32
            pending = cur.scale is not None or cur.residual is not None or cur.act != ACT_NONE
            if not self.switches.fuse_residual and pending:
                # separate skip-add pass: materialise r_b once, the first conv then loads it unchanged
                r = self._apply(cur.x, cur.scale, cur.shift, cur.act, residual=cur.residual, want_f32=True, want_split=False).f32
                cur = Lazy(r)
                pending = False
            y, ws, r = self._consume(cv1, cur, N, h, w, pad=bpad, border=b, keep=pending, block=True)
            if r is None:
                r = cur.x
            sc, sh = self._stats(y, nm1, ws)
            y, ws, _ = self._consume(cv2, Lazy(y, sc, sh, ACT_RELU), N, h, w, pad=bpad, border=b, block=True)
            sc, sh = self._stats(y, nm2, ws)
            cur = Lazy(y, sc, sh, ACT_NONE, residual=r)
            tap(f"block{bi}", cur)
        for i in range(2):
            y, ws, _ = self._consume(self.up[i], cur, N, h, w, allow=(2, 4) if self.switches.fuse_up else ())
            h, w = h * 2, w * 2
            sc, sh = self._stats(y, self.up_norm[i], ws)
            cur = Lazy(y, sc, sh, ACT_RELU)
        if plan.head == "stream":
            return ops.head_conv(cur.x, cur.scale, cur.shift, cur.act, self.head_wpk, self.head_bias, self.head_co, self.pad_mode,
                                 ACT_TANH)
        z, _, _ = self._consume(self.head, cur, N, h, w, border=3, fuse_stats=False, allow=(1, 2) if self.switches.fuse_head else ())
        return ops.head_finish(z, self.head_bias, w, self.head_S, self.head_co, ACT_TANH)

    __call__ = forward


def _pad_cout32(w, transposed):
    """Zero-pad the output-channel dim of a conv weight to 32 so a Cout <= 4 layer fits a tensor-core tile."""
    if transposed:
        ci, co, R, S = w.shape
        out = torch.zeros((ci, 32, R, S), dtype=torch.float32, device=w.device)
        out[:, :co] = w
    else:
        co, ci, R, S = w.shape
        out = torch.zeros((32, ci, R, S), dtype=torch.float32, device=w.device)
        out[:co] = w
    return out, co


class UnetEngine(_EngineBase):
    """UnetGenerator forward (eval semantics).  Level k (0 = outermost) follows UnetSkipConnectionBlock
    (networks.py:573-615): down = [LeakyReLU(0.2), Conv4x4 s2, Norm], up = [ReLU, ConvT4x4 s2, Norm], skip =
    cat([x, model(x)], 1).  The skip concat is never materialised: every up-convolution reads its two sources
    (skip, below) through two TMA tensor maps (dual-source K loop); relu(cat(a, u)) = cat(relu(a), relu(u)) and
    relu(leaky_relu(x)) = relu(x), so the skip operand is relu(norm(d_{k-1}))."""

    def __init__(self, sd, *, num_downs=9, norm="batch", norm_mode="sample", precision="bf16x3", backend="tc",
                 device="cuda"):
        prec = Precision.parse(precision) if isinstance(precision, str) else precision
        super().__init__(norm, norm_mode, prec, backend, device)
        if backend != "tc":
            raise NotImplementedError("UnetEngine runs on the tensor-core backend only")
        self.nd = num_downs
        g = lambda k: sd[k].to(device) if k in sd else None
        pre = ["model.model"]
        for lvl in range(1, num_downs):
            pre.append(f"{pre[-1]}.{1 if lvl == 1 else 3}.model")
        self.down, self.down_norm, self.up, self.up_norm = [], [], [], []
        for lvl in range(num_downs):
            p = pre[lvl]
            innermost = lvl == num_downs - 1
            dk = f"{p}.0" if lvl == 0 else f"{p}.1"
            uk = f"{p}.3" if (lvl == 0 or innermost) else f"{p}.5"
            self.down.append(ConvLayer(g(dk + ".weight"), g(dk + ".bias"), stride=2, pad=1, prec=prec, backend=backend))
            self.down_norm.append(_NormParams(sd, f"{p}.2", norm, device) if (0 < lvl < num_downs - 1) else None)
            wu, bu = g(uk + ".weight").to(torch.float32), g(uk + ".bias")
            cin_total, cout = wu.shape[0], wu.shape[1]
            cins = [cin_total] if innermost else [cin_total // 2, cin_total // 2]
            if lvl == 0:
                if cout > 4:
                    raise NotImplementedError("UnetEngine: output_nc <= 4 expected")
                wu, self.out_nc = _pad_cout32(wu, True)
                self.out_bias = bu.detach().to(torch.float32).contiguous()
                self.up.append(ConvLayer(wu, None, transposed=True, stride=2, pad=1, cins=cins, prec=prec, backend="tc",
                                         n_tile=32))
            else:
                self.up.append(ConvLayer(wu, bu, transposed=True, stride=2, pad=1, cins=cins, prec=prec, backend="tc"))
            nk = None if lvl == 0 else (f"{p}.4" if innermost else f"{p}.6")
            self.up_norm.append(_NormParams(sd, nk, norm, device) if nk else None)

    @torch.no_grad()
    def forward(self, x, taps=None):
        x = x.contiguous()
        N, _, H, W = x.shape
        nd = self.nd
        # ---- down path: keep, per level, the raw conv output + its (scale, shift) ---------------------------------
        raw, ss = [], []
        h, w = H, W
        y = self.down[0].run_direct(x, N, h, w, in_nchw=True)             # level 0: Conv(input_nc -> ngf), no norm
        h, w = h // 2, w // 2
        raw.append(y); ss.append((None, None))
        dims = [(h, w)]
        for lvl in range(1, nd):
            sc, sh = ss[-1]
            a = self._apply(raw[-1], sc, sh, ACT_LRELU02)                  # LeakyReLU(0.2)(norm(d_{lvl-1}))
            y, ws = self.down[lvl].run_tc([a], N, h, w)
            h, w = h // 2, w // 2
            raw.append(y)
            ss.append(self._stats(y, self.down_norm[lvl], ws) if self.down_norm[lvl] is not None else (None, None))
            dims.append((h, w))
        # ---- up path --------------------------------------------------------------------------------------------------
        # relu(norm(.)) of the skip and of the level below are evaluated by the up-convolution itself while it loads its
        # two K-sources (fused operand, halo-strip mode) wherever the map is at least 16 x 8; below that one
        # dlb_norm_apply pass per source writes the operand planes.
        fused = _env_flag("DLB_FUSED", True)
        below = None                                                       # Lazy: raw up-conv output + its (scale, shift)
        for lvl in range(nd - 1, -1, -1):
            h, w = dims[lvl]
            sc, sh = ss[lvl]
            lz = [Lazy(raw[lvl], sc, sh, ACT_RELU)] + ([] if lvl == nd - 1 else [below])   # relu of both skip halves
            layer = self.up[lvl]
            use_fused = fused and ops.conv_tc_fused_mode(layer.desc(N, h, w), self.prec.split, layer.n_tile) == 2
            if use_fused:
                run = lambda fs: layer.run_fused([l.src() for l in lz], N, h, w, fuse_stats=fs)
            else:
                acts = [self._apply(l.x, l.scale, l.shift, l.act) for l in lz]
                run = lambda fs: layer.run_tc(acts, N, h, w, fuse_stats=fs)
            if lvl == 0:
                z, _ = run(False)
                return ops.head_finish(z, self.out_bias, 2 * w, 1, self.out_nc, ACT_TANH)
            y, ws = run(True)
            usc, ush = self._stats(y, self.up_norm[lvl], ws)
            below = Lazy(y, usc, ush, ACT_RELU)                             # relu(norm(u_lvl)) for the level above
            if taps is not None:
                taps[f"up{lvl}"] = below

    __call__ = forward


class NLayerDEngine(_EngineBase):
    """NLayerDiscriminator forward (networks.py:636-660): Conv4x4 s2 (+bias) LReLU; [Conv4x4 s2, Norm, LReLU] x (n-1);
    Conv4x4 s1, Norm, LReLU; Conv4x4 s1 (-> 1, +bias).  Training-time module: norm_mode defaults to 'batch'."""

    def __init__(self, sd, *, n_layers=3, norm="batch", norm_mode="batch", precision="bf16x3", backend="tc",
                 device="cuda"):
        prec = Precision.parse(precision) if isinstance(precision, str) else precision
        super().__init__(norm, norm_mode, prec, backend, device)
        g = lambda k: sd[k].to(device) if k in sd else None
        # first conv: Cin = 6 padded to 64 zero lanes so it runs (forward, wgrad, dgrad) on the tensor cores
        w0 = g("model.0.weight").to(torch.float32)
        w0p = torch.zeros((w0.shape[0], 64, w0.shape[2], w0.shape[3]), dtype=torch.float32, device=device)
        w0p[:, : w0.shape[1]] = w0
        self.first = ConvLayer(w0p, g("model.0.bias"), stride=2, pad=1, prec=prec, backend="tc")
        self.mid = []
        idx = 2
        for n in range(1, n_layers + 1):
            st = 2 if n < n_layers else 1
            self.mid.append((ConvLayer(g(f"model.{idx}.weight"), g(f"model.{idx}.bias"), stride=st, pad=1, prec=prec,
                                       backend=backend), _NormParams(sd, f"model.{idx + 1}", norm, device)))
            idx += 3
        wl, bl = g(f"model.{idx}.weight").to(torch.float32), g(f"model.{idx}.bias")
        wl32, self.out_nc = _pad_cout32(wl, False)
        self.last = ConvLayer(wl32, None, stride=1, pad=1, prec=prec, backend="tc", n_tile=32)
        self.last_bias = bl.detach().to(torch.float32).contiguous()

    @torch.no_grad()
    def forward(self, x, taps=None):
        """x: fp32 NCHW [N, 6, H, W] (cat of condition and image) -> fp32 NCHW [N, 1, h, w] logits."""
        x = x.contiguous()
        N, _, H, W = x.shape
        xh, xl = ops.stem_window_pack(x, 0, 1, PAD_ZERO, self.prec.fmt, self.prec.split)
        y, _ = self.first.run_tc([Act(None, xh, xl)], N, H, W, fuse_stats=False)
        h, w = H // 2, W // 2
        sc = sh = None
        for cv, nm in self.mid:
            a = self._apply(y, sc, sh, ACT_LRELU02)
            y, ws = cv.run_tc([a], N, h, w)
            h, w = y.shape[1], y.shape[2]
            sc, sh = self._stats(y, nm, ws)
        a = self._apply(y, sc, sh, ACT_LRELU02)
        z, _ = self.last.run_tc([a], N, h, w, fuse_stats=False)
        return ops.head_finish(z, self.last_bias, z.shape[2], 1, self.out_nc, ACT_NONE)

    __call__ = forward
