"""Thin torch-tensor wrappers over the C ABI (include/deepliif_b200.h).

PyTorch is used for device memory (caching allocator) and streams only; every wrapper enqueues exactly the
library call on torch's current CUDA stream.  No wrapper has a PyTorch-op fallback.
"""
import ctypes as C

import torch

from . import _lib
from ._lib import (ACT_LRELU02, ACT_NONE, ACT_RELU, ACT_TANH, FMT_BF16, FMT_FP16, PAD_REFLECT, PAD_ZERO,
                   ConvDesc, FusedSrc, check)

__all__ = ["ConvDesc", "conv_desc", "conv_out_shape", "pack_weights_tc", "pack_weights_direct", "conv_tc", "conv_tc_fused", "conv_tc_fused_mode", "conv_tc_stem",
           "conv_direct", "norm_stats", "norm_finalize", "stats_workspace", "norm_bwd", "conv_wgrad", "head_bwd_pack", "channel_sum", "adam_step", "adam_hyper", "adam_step_dev", "norm_apply", "stem_window_pack", "reflect_fold", "stem_window_bwd", "head_finish", "head_conv", "head_conv_pack", "stem_conv", "stem_conv_pack", "tile_gray_variance", "u8_to_f32", "f32_to_u8", "seg_finish", "LAUNCHES",
           "FMT_BF16", "FMT_FP16", "ACT_NONE", "ACT_RELU", "ACT_LRELU02", "ACT_TANH", "PAD_ZERO", "PAD_REFLECT"]

# kernel-launch counter (bench.py reports gpu_launches from this)
LAUNCHES = {"count": 0}


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _raw_stream():
    """Handle of torch's current CUDA stream (the C-level getter: torch.cuda.current_stream() builds a Stream object
    and costs ~10 us, which adds up over the ~2000 launches of a training step)."""
    return torch._C._cuda_getCurrentRawStream(torch._C._cuda_getDevice())


def _stream():
    return C.c_void_p(_raw_stream())


def _dtype(fmt):
    return torch.bfloat16 if fmt == FMT_BF16 else torch.float16


def _need_cuda(*ts):
    for t in ts:
        if t is not None and (not t.is_cuda or not t.is_contiguous()):
            raise _lib.DeepliifB200Error("deepliif_b200 ops need contiguous CUDA tensors (no CPU path exists)")


def _need_shape(what, t, shape):
    """A tensor the kernel would index by the descriptor's extents must have exactly those extents: a mismatch is
    refused here, before anything is launched."""
    if t is not None and tuple(t.shape) != tuple(shape):
        raise _lib.DeepliifB200Error(f"{what}: tensor of shape {tuple(t.shape)}, the descriptor needs {tuple(shape)}")


def conv_desc(N, H, W, cins, Cout, R, S, stride=1, pad=0, transposed=False, output_padding=0, pad_mode=PAD_ZERO):
    cins = list(cins) if isinstance(cins, (list, tuple)) else [cins]
    arr = (C.c_int * 2)(*(cins + [0] * (2 - len(cins))))
    return ConvDesc(N, H, W, len(cins), arr, Cout, R, S, stride, pad, int(transposed), output_padding, pad_mode)


def conv_out_shape(d):
    oh, ow = C.c_int(), C.c_int()
    check(_lib.load().dlb_conv_out_shape(C.byref(d), C.byref(oh), C.byref(ow)), "dlb_conv_out_shape")
    return oh.value, ow.value


def _cin_total(d):
    return sum(d.Cin[i] for i in range(d.nsrc))


def pack_weights_tc(d, w, fmt=FMT_BF16, split=True):
    """w: fp32 CUDA, Conv2d (Cout,Cin,R,S) or ConvTranspose2d (Cin,Cout,R,S) -> (hi, lo) [R*S, Cout, Cin]."""
    _need_cuda(w)
    shape = (d.R * d.S, d.Cout, _cin_total(d))
    hi = torch.empty(shape, dtype=_dtype(fmt), device=w.device)
    lo = torch.empty(shape, dtype=_dtype(fmt), device=w.device) if split else None
    check(_lib.load().dlb_pack_weights_tc(C.byref(d), _p(w), fmt, _p(hi), _p(lo), _stream()), "dlb_pack_weights_tc")
    LAUNCHES["count"] += 1
    return hi, lo


def pack_weights_direct(d, w):
    _need_cuda(w)
    out = torch.empty((d.R * d.S, _cin_total(d), d.Cout), dtype=torch.float32, device=w.device)
    check(_lib.load().dlb_pack_weights_direct(C.byref(d), _p(w), _p(out), _stream()), "dlb_pack_weights_direct")
    LAUNCHES["count"] += 1
    return out


_WS_CACHE = {}


def stats_workspace(N, HW, C, device):
    """Zero-initialised statistics workspace (cached per shape/device; calls leave it clean)."""
    key = (N, HW, C, str(device), _raw_stream())   # one workspace per stream
    ws = _WS_CACHE.get(key)
    if ws is None:
        nbytes = _lib.load().dlb_norm_stats_workspace(N, HW, C)
        ws = torch.zeros((nbytes + 3) // 4, dtype=torch.float32, device=device)
        _WS_CACHE[key] = ws
    return ws


def conv_tc(d, xs_hi, xs_lo, w_hi, w_lo, bias=None, fmt=FMT_BF16, split=True, n_tile=0, out=None, stats_ws=None):
    """Tensor-core conv.  xs_hi/xs_lo: lists (one per source) of NHWC 16-bit planes.  Returns fp32 NHWC.
    stats_ws: workspace from stats_workspace(N, OH*OW, Cout) -> the epilogue also emits partial statistics."""
    xs_hi = list(xs_hi) if isinstance(xs_hi, (list, tuple)) else [xs_hi]
    xs_lo = (list(xs_lo) if isinstance(xs_lo, (list, tuple)) else [xs_lo]) if split else [None] * len(xs_hi)
    _need_cuda(*xs_hi, *xs_lo, w_hi, w_lo, bias)
    if len(xs_hi) != d.nsrc:
        raise _lib.DeepliifB200Error(f"conv_tc: {len(xs_hi)} sources, the descriptor has {d.nsrc}")
    for s_, (xh, xl) in enumerate(zip(xs_hi, xs_lo)):
        _need_shape(f"conv_tc source {s_}", xh, (d.N, d.H, d.W, d.Cin[s_]))
        _need_shape(f"conv_tc source {s_} (lo)", xl, (d.N, d.H, d.W, d.Cin[s_]))
    oh, ow = conv_out_shape(d)
    if out is None:
        out = torch.empty((d.N, oh, ow, d.Cout), dtype=torch.float32, device=w_hi.device)
    hi_arr = (C.c_void_p * 2)(*[x.data_ptr() for x in xs_hi] + [None] * (2 - len(xs_hi)))
    lo_arr = (C.c_void_p * 2)(*[(x.data_ptr() if x is not None else None) for x in xs_lo] + [None] * (2 - len(xs_lo)))
    check(_lib.load().dlb_conv_tc_fwd(C.byref(d), hi_arr, lo_arr, _p(w_hi), _p(w_lo) if split else None, _p(bias),
                                      _p(out), fmt, int(split), n_tile, _p(stats_ws),
                                      stats_ws.numel() * 4 if stats_ws is not None else 0, _stream()),
          "dlb_conv_tc_fwd")
    LAUNCHES["count"] += _lib.load().dlb_conv_tc_launches(C.byref(d), int(split), n_tile, 0) if d.transposed else 1
    return out


def conv_tc_fused_mode(d, split=True, n_tile=0):
    """2 / 1: the fused-operand kernel runs this layer in a strip mode (efficient); 0: it would convert per tap."""
    m = _lib.load().dlb_conv_tc_fused_mode(C.byref(d), int(split), n_tile)
    if m < 0:
        check(m, "dlb_conv_tc_fused_mode")
    return m


def conv_tc_fused(d, srcs, w_hi, w_lo, bias=None, fmt=FMT_BF16, split=True, n_tile=0, out=None, stats_ws=None):
    """Tensor-core conv whose operand is evaluated inside the kernel from the producer's raw fp32 output.
    srcs: one dict per K-source with keys x (fp32 NHWC), scale, shift ([N,C] or None), act, residual (fp32 NHWC or None),
    out (fp32 NHWC or None: receives the evaluated operand), border, border_mode.  d.H / d.W include 2*border."""
    arr = (FusedSrc * 2)()
    keep = []
    if len(srcs) != d.nsrc:
        raise _lib.DeepliifB200Error(f"conv_tc_fused: {len(srcs)} sources, the descriptor has {d.nsrc}")
    for i, s_ in enumerate(srcs):
        x, sc, sh, res, o = s_["x"], s_.get("scale"), s_.get("shift"), s_.get("residual"), s_.get("out")
        _need_cuda(x, sc, sh, res, o)
        if x.dtype != torch.float32:
            raise _lib.DeepliifB200Error("conv_tc_fused: sources are fp32 NHWC tensors")
        bd = int(s_.get("border", 0))
        shape = (d.N, d.H - 2 * bd, d.W - 2 * bd, d.Cin[i])
        for what, t in (("x", x), ("residual", res), ("out", o)):
            _need_shape(f"conv_tc_fused source {i} {what}", t, shape)
        keep += [x, sc, sh, res, o]
        arr[i] = FusedSrc(x.data_ptr(), sc.data_ptr() if sc is not None else None, sh.data_ptr() if sh is not None else None,
                          int(s_.get("act", ACT_NONE)), res.data_ptr() if res is not None else None,
                          o.data_ptr() if o is not None else None, int(s_.get("border", 0)), int(s_.get("border_mode", PAD_ZERO)))
    _need_cuda(w_hi, w_lo, bias)
    oh, ow = conv_out_shape(d)
    if out is None:
        out = torch.empty((d.N, oh, ow, d.Cout), dtype=torch.float32, device=w_hi.device)
    check(_lib.load().dlb_conv_tc_fwd_fused(C.byref(d), arr, _p(w_hi), _p(w_lo) if split else None, _p(bias), _p(out), fmt,
                                            int(split), n_tile, _p(stats_ws),
                                            stats_ws.numel() * 4 if stats_ws is not None else 0, _stream()),
          "dlb_conv_tc_fwd_fused")
    LAUNCHES["count"] += _lib.load().dlb_conv_tc_launches(C.byref(d), int(split), n_tile, 1) if d.transposed else 1
    return out


def conv_tc_stem(x_nchw, pad, S, pad_mode, cout, w_hi, w_lo, bias=None, fmt=FMT_BF16, split=True, n_tile=0, stats_ws=None):
    """Pad(pad) + Conv2d(C <= 4 -> cout, S x S) from the fp32 NCHW input in one tensor-core kernel (the window operand is
    built in shared memory).  w_hi / w_lo: planes of the 64-lane vertical weight (see dlb_stem_window_pack).  fp32 NHWC out."""
    _need_cuda(x_nchw, w_hi, w_lo, bias)
    N, Cc, H, W = x_nchw.shape
    out = torch.empty((N, H, W, cout), dtype=torch.float32, device=x_nchw.device)
    check(_lib.load().dlb_conv_tc_fwd_stem(_p(x_nchw), N, Cc, H, W, pad, S, pad_mode, cout, _p(w_hi), _p(w_lo) if split else None,
                                           _p(bias), _p(out), fmt, int(split), n_tile, _p(stats_ws),
                                           stats_ws.numel() * 4 if stats_ws is not None else 0, _stream()),
          "dlb_conv_tc_fwd_stem")
    LAUNCHES["count"] += 1
    return out


def conv_direct(d, x, w_packed, bias=None, in_nchw=False, in_scale=None, in_shift=None, in_act=ACT_NONE,
                out_act=ACT_NONE, out_nchw=False, out=None):
    _need_cuda(x, w_packed, bias, in_scale, in_shift)
    cin = _cin_total(d)
    _need_shape("conv_direct x", x, (d.N, cin, d.H, d.W) if in_nchw else (d.N, d.H, d.W, cin))
    oh, ow = conv_out_shape(d)
    if out is None:
        shape = (d.N, d.Cout, oh, ow) if out_nchw else (d.N, oh, ow, d.Cout)
        out = torch.empty(shape, dtype=torch.float32, device=x.device)
    check(_lib.load().dlb_conv_direct_fwd(C.byref(d), _p(x), int(in_nchw), _p(in_scale), _p(in_shift), in_act,
                                          _p(w_packed), _p(bias), _p(out), out_act, int(out_nchw), _stream()),
          "dlb_conv_direct_fwd")
    LAUNCHES["count"] += (d.stride * d.stride if d.transposed else 1)
    return out


def norm_finalize(ws, N, HW, Cc, gamma=None, beta=None, pooled=False, eps=1e-5, want_stats=False, running=None):
    """Reduce the partial statistics a conv epilogue left in `ws` -> (scale, shift) fp32 [N,C]
    (+ (mean, rstd) with want_stats, kept for the backward pass).  running = (running_mean, running_var,
    num_batches_tracked, momentum): training-mode BatchNorm2d buffers, updated in the same kernel (pooled only)."""
    scale = torch.empty((N, Cc), dtype=torch.float32, device=ws.device)
    shift = torch.empty((N, Cc), dtype=torch.float32, device=ws.device)
    mean = torch.empty((N, Cc), dtype=torch.float32, device=ws.device) if want_stats else None
    rstd = torch.empty((N, Cc), dtype=torch.float32, device=ws.device) if want_stats else None
    if running is not None and pooled:
        rm, rv, nbt, mom = running
        _need_cuda(rm, rv, nbt)
        check(_lib.load().dlb_norm_finalize_bn(_p(ws), ws.numel() * 4, N, HW, Cc, _p(gamma), _p(beta), float(eps), _p(scale),
                                               _p(shift), _p(mean), _p(rstd), _p(rm), _p(rv), _p(nbt), float(mom), _stream()),
              "dlb_norm_finalize_bn")
        LAUNCHES["count"] += 1
        return (scale, shift, mean, rstd) if want_stats else (scale, shift)
    check(_lib.load().dlb_norm_finalize(_p(ws), ws.numel() * 4, N, HW, Cc, int(pooled), _p(gamma), _p(beta),
                                        float(eps), _p(scale), _p(shift), _p(mean), _p(rstd), _stream()), "dlb_norm_finalize")
    LAUNCHES["count"] += 1
    return (scale, shift, mean, rstd) if want_stats else (scale, shift)


def norm_stats(y, gamma=None, beta=None, pooled=False, eps=1e-5, want_stats=False, running=None):
    """y: fp32 NHWC [N,H,W,C] -> (scale, shift) fp32 [N,C] with norm(y) = y*scale + shift (+ mean, rstd).
    running: see norm_finalize."""
    _need_cuda(y, gamma, beta)
    N, H, W, Cc = y.shape
    lib = _lib.load()
    ws = stats_workspace(N, H * W, Cc, y.device)
    ws_bytes = ws.numel() * 4
    scale = torch.empty((N, Cc), dtype=torch.float32, device=y.device)
    shift = torch.empty((N, Cc), dtype=torch.float32, device=y.device)
    mean = torch.empty((N, Cc), dtype=torch.float32, device=y.device) if want_stats else None
    rstd = torch.empty((N, Cc), dtype=torch.float32, device=y.device) if want_stats else None
    if running is not None and pooled:
        rm, rv, nbt, mom = running
        _need_cuda(rm, rv, nbt)
        check(lib.dlb_norm_stats_bn(_p(y), N, H * W, Cc, _p(gamma), _p(beta), float(eps), _p(scale), _p(shift), _p(mean),
                                    _p(rstd), _p(rm), _p(rv), _p(nbt), float(mom), _p(ws), ws_bytes, _stream()),
              "dlb_norm_stats_bn")
    else:
        check(lib.dlb_norm_stats(_p(y), N, H * W, Cc, int(pooled), _p(gamma), _p(beta), float(eps), _p(scale), _p(shift),
                                 _p(mean), _p(rstd), _p(ws), ws_bytes, _stream()), "dlb_norm_stats")
    LAUNCHES["count"] += 2
    return (scale, shift, mean, rstd) if want_stats else (scale, shift)


def norm_bwd(dout, y, scale=None, shift=None, mean=None, rstd=None, act=ACT_NONE, dout2=None, act2=None, pooled=False,
             dgamma=None, dbeta=None, accumulate=False, want_f32=False, want_split=True, fmt=FMT_BF16, need_lo=True,
             drop_p=0.0, drop_seed=0, drop_epoch=None):
    """Backward of norm(+affine)+activation: returns (dy_f32 | None, dy_hi | None, dy_lo | None); writes the
    parameter gradients into dgamma/dbeta (fp32 [C]) when given.  scale=None: layer without norm."""
    _need_cuda(dout, dout2, y, scale, shift, mean, rstd, dgamma, dbeta)
    N, H, W, Cc = y.shape
    dev = y.device
    c1 = torch.empty((N, Cc), dtype=torch.float32, device=dev) if scale is not None else None
    c2 = torch.empty((N, Cc), dtype=torch.float32, device=dev) if scale is not None else None
    f32 = torch.empty_like(y) if want_f32 else None
    hi = torch.empty(y.shape, dtype=_dtype(fmt), device=dev) if want_split else None
    lo = torch.empty(y.shape, dtype=_dtype(fmt), device=dev) if (want_split and need_lo) else None
    ws = stats_workspace(N, H * W, Cc, dev)
    check(_lib.load().dlb_norm_bwd(_p(dout), _p(dout2), _p(y), _p(scale), _p(shift), _p(mean), _p(rstd), act,
                                   act if act2 is None else act2, N, H * W, Cc,
                                   int(pooled), _p(c1), _p(c2), _p(dgamma), _p(dbeta), int(accumulate), _p(f32), _p(hi),
                                   _p(lo), fmt, float(drop_p), int(drop_seed), _p(drop_epoch), _p(ws), ws.numel() * 4, _stream()),
          "dlb_norm_bwd")
    LAUNCHES["count"] += 3 if scale is not None else 1
    return f32, hi, lo


_WG_CACHE = {}


def adam_hyper(lr, beta1, beta2, step, grad_scale=1.0):
    """The four step-dependent floats of the update, computed by the library (same arithmetic as dlb_adam_step)."""
    buf = (C.c_float * 4)()
    check(_lib.load().dlb_adam_hyper(float(lr), float(beta1), float(beta2), int(step), float(grad_scale), buf), "dlb_adam_hyper")
    return list(buf)


def adam_step_dev(p, g, m, v, hyper_dev, beta1, beta2, eps):
    """Fused Adam with {lr, bc1, sqrt(bc2), grad_scale} read from the device tensor hyper_dev (graph-capturable)."""
    _need_cuda(p, g, m, v, hyper_dev)
    check(_lib.load().dlb_adam_step_dev(_p(p), _p(g), _p(m), _p(v), p.numel(), _p(hyper_dev), float(beta1), float(beta2),
                                        float(eps), _stream()), "dlb_adam_step_dev")
    LAUNCHES["count"] += 1


def adam_step(p, g, m, v, lr, beta1, beta2, eps, step, grad_scale=1.0):
    """In-place fused Adam on flat fp32 buffers."""
    _need_cuda(p, g, m, v)
    check(_lib.load().dlb_adam_step(_p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(beta1), float(beta2), float(eps),
                                    int(step), float(grad_scale), _stream()), "dlb_adam_step")
    LAUNCHES["count"] += 1


def channel_sum(x, out=None, accumulate=False):
    """Sum over all leading dims of fp32 [..., C] -> [C] (bias gradient)."""
    _need_cuda(x, out)
    Cc = x.shape[-1]
    rows = x.numel() // Cc
    key = ("chsum", Cc, str(x.device), _raw_stream())
    ws = _WG_CACHE.get(key)
    if ws is None:
        ws = _WG_CACHE[key] = torch.empty(1024 * Cc, dtype=torch.float32, device=x.device)
    if out is None:
        out = torch.empty(Cc, dtype=torch.float32, device=x.device)
        accumulate = False
    check(_lib.load().dlb_channel_sum(_p(x), rows, Cc, _p(out), int(accumulate), _p(ws), ws.numel() * 4, _stream()),
          "dlb_channel_sum")
    LAUNCHES["count"] += 2
    return out


def conv_wgrad(d, x_hi, x_lo, dy_hi, dy_lo, dw=None, accumulate=False, fmt=FMT_BF16, split=True):
    """Weight gradient (fp32, PyTorch weight layout) of the forward layer `d` from hi/lo NHWC planes."""
    _need_cuda(x_hi, x_lo, dy_hi, dy_lo, dw)
    lib = _lib.load()
    nbytes = lib.dlb_conv_wgrad_workspace(C.byref(d))
    if nbytes == 0:
        check(-1, "dlb_conv_wgrad_workspace")
    key = (nbytes, str(x_hi.device), _raw_stream())
    ws = _WG_CACHE.get(key)
    if ws is None:
        ws = _WG_CACHE[key] = torch.empty((nbytes + 3) // 4, dtype=torch.float32, device=x_hi.device)
    if dw is None:
        cin = _cin_total(d)
        shape = (cin, d.Cout, d.R, d.S) if d.transposed else (d.Cout, cin, d.R, d.S)
        dw = torch.empty(shape, dtype=torch.float32, device=x_hi.device)
        accumulate = False
    check(lib.dlb_conv_wgrad(C.byref(d), _p(x_hi), _p(x_lo) if split else None, _p(dy_hi), _p(dy_lo) if split else None,
                             _p(dw), int(accumulate), fmt, int(split), _p(ws), ws.numel() * 4, _stream()), "dlb_conv_wgrad")
    LAUNCHES["count"] += 2
    return dw


def head_bwd_pack(dzz_nchw, S, fmt=FMT_BF16, need_lo=True):
    """dzz fp32 NCHW [N,CO<=4,H,W] -> (hi, lo) planes [N, H, W+S-1, 64] with lane j = s*4 + co."""
    _need_cuda(dzz_nchw)
    N, CO, H, W = dzz_nchw.shape
    shp = (N, H, W + S - 1, 64)
    hi = torch.empty(shp, dtype=_dtype(fmt), device=dzz_nchw.device)
    lo = torch.empty(shp, dtype=_dtype(fmt), device=dzz_nchw.device) if need_lo else None
    check(_lib.load().dlb_head_bwd_pack(_p(dzz_nchw), N, H, W, S, CO, fmt, _p(hi), _p(lo), _stream()), "dlb_head_bwd_pack")
    LAUNCHES["count"] += 1
    return hi, lo


def norm_apply(y, scale=None, shift=None, act=ACT_NONE, residual=None, want_f32=False, want_split=True,
               fmt=FMT_BF16, pad=0, pad_mode=PAD_ZERO, need_lo=True, drop_p=0.0, drop_seed=0, drop_epoch=None):
    """out = act(y*scale+shift) (+ residual) -> (out_f32 | None, hi | None, lo | None)."""
    _need_cuda(y, scale, shift, residual)
    N, H, W, Cc = y.shape
    _need_shape("norm_apply scale", scale, (N, Cc))
    _need_shape("norm_apply shift", shift, (N, Cc))
    _need_shape("norm_apply residual", residual, y.shape)
    f32 = torch.empty_like(y) if want_f32 else None
    hi = lo = None
    if want_split:
        shp = (N, H + 2 * pad, W + 2 * pad, Cc)
        hi = torch.empty(shp, dtype=_dtype(fmt), device=y.device)
        lo = torch.empty(shp, dtype=_dtype(fmt), device=y.device) if need_lo else None
    check(_lib.load().dlb_norm_apply(_p(y), _p(scale), _p(shift), act, _p(residual), _p(f32), _p(hi), _p(lo), fmt,
                                     N, H, W, Cc, pad, pad_mode, float(drop_p), int(drop_seed), _p(drop_epoch), _stream()),
          "dlb_norm_apply")
    LAUNCHES["count"] += 1
    return f32, hi, lo


def reflect_fold(dpad, pad, add=None):
    """Backward of ReflectionPad2d(pad): dpad fp32 [N,H+2p,W+2p,C] (+ add [N,H,W,C]) -> fp32 [N,H,W,C]."""
    _need_cuda(dpad, add)
    N, HP, WP, Cc = dpad.shape
    H, W = HP - 2 * pad, WP - 2 * pad
    out = torch.empty((N, H, W, Cc), dtype=torch.float32, device=dpad.device)
    check(_lib.load().dlb_reflect_fold(_p(dpad), _p(add), N, H, W, Cc, pad, _p(out), _stream()), "dlb_reflect_fold")
    LAUNCHES["count"] += 1
    return out


def stem_window_bwd(dxw, C, pad, S, pad_mode=PAD_ZERO):
    """Backward of stem_window_pack: dxw fp32 [N,H+2p,W,64] -> dx fp32 NCHW [N,C,H,W]."""
    _need_cuda(dxw)
    N, HP, W, lanes = dxw.shape
    assert lanes == 64
    H = HP - 2 * pad
    dx = torch.empty((N, C, H, W), dtype=torch.float32, device=dxw.device)
    check(_lib.load().dlb_stem_window_bwd(_p(dxw), N, C, H, W, pad, S, pad_mode, _p(dx), _stream()), "dlb_stem_window_bwd")
    LAUNCHES["count"] += 1
    return dx


def stem_window_pack(x_nchw, pad, S, pad_mode=PAD_ZERO, fmt=FMT_BF16, need_lo=True):
    """x fp32 NCHW [N,C<=8,H,W] -> (hi, lo) planes [N, H+2pad, W, 64] with k = s*8 + c (see include)."""
    _need_cuda(x_nchw)
    N, Cc, H, W = x_nchw.shape
    shp = (N, H + 2 * pad, W, 64)
    hi = torch.empty(shp, dtype=_dtype(fmt), device=x_nchw.device)
    lo = torch.empty(shp, dtype=_dtype(fmt), device=x_nchw.device) if need_lo else None
    check(_lib.load().dlb_stem_window_pack(_p(x_nchw), N, Cc, H, W, pad, S, pad_mode, fmt, _p(hi), _p(lo), _stream()),
          "dlb_stem_window_pack")
    LAUNCHES["count"] += 1
    return hi, lo


def head_finish(z, bias, W, S, CO, act=ACT_TANH):
    """z fp32 NHWC [N,H,W+S-1,32] -> fp32 NCHW [N,CO,H,W] (shifted tap sum + bias + activation)."""
    _need_cuda(z, bias)
    N, H, WZ, _ = z.shape
    assert WZ == W + S - 1 and z.shape[3] == 32
    out = torch.empty((N, CO, H, W), dtype=torch.float32, device=z.device)
    check(_lib.load().dlb_head_finish(_p(z), _p(bias), N, H, W, S, CO, act, _p(out), _stream()), "dlb_head_finish")
    LAUNCHES["count"] += 1
    return out


def stem_conv_pack(w):
    """w fp32 [64, C<=4, 7, 7] (PyTorch layout) -> the packed split-precision weight image of dlb_stem_conv_fwd."""
    w = w.detach().to(torch.float32).contiguous()
    _need_cuda(w)
    co, ci, R, S = w.shape
    lib = _lib.load()
    out = torch.empty((lib.dlb_stem_conv_weight_bytes(),), dtype=torch.uint8, device=w.device)
    check(lib.dlb_stem_conv_pack_weights(_p(w), co, ci, R, S, _p(out), _stream()), "dlb_stem_conv_pack_weights")
    LAUNCHES["count"] += 1
    return out


def stem_conv(x_nchw, w_packed, bias, cout, border_mode, stats_ws=None):
    """Pad(3) + Conv2d(C <= 4 -> 64, 7) (+ bias) from the fp32 NCHW input; fp32 NHWC [N, H, W, 64] out and, with stats_ws,
    the partial statistics for norm_finalize.  One row-streaming tensor-core kernel (dlb_stem_conv_fwd)."""
    _need_cuda(x_nchw, w_packed, bias)
    N, Cc, H, W = x_nchw.shape
    out = torch.empty((N, H, W, cout), dtype=torch.float32, device=x_nchw.device)
    check(_lib.load().dlb_stem_conv_fwd(_p(x_nchw), N, Cc, H, W, _p(w_packed), _p(bias), cout, border_mode, _p(out), _p(stats_ws),
                                        stats_ws.numel() * 4 if stats_ws is not None else 0, _stream()), "dlb_stem_conv_fwd")
    LAUNCHES["count"] += 1
    return out


def head_conv_pack(w):
    """w fp32 [CO<=3, 64, 7, 7] (PyTorch layout) -> the packed split-precision weight image of dlb_head_conv_fwd."""
    w = w.detach().to(torch.float32).contiguous()
    _need_cuda(w)
    co, ci, R, S = w.shape
    lib = _lib.load()
    out = torch.empty((lib.dlb_head_conv_weight_bytes(),), dtype=torch.uint8, device=w.device)
    check(lib.dlb_head_conv_pack_weights(_p(w), co, ci, R, S, _p(out), _stream()), "dlb_head_conv_pack_weights")
    LAUNCHES["count"] += 1
    return out


def head_conv(x, scale, shift, act, w_packed, bias, CO, border_mode, out_act=ACT_TANH):
    """Pad(3) + Conv2d(64 -> CO, 7) + bias + activation on act(x*scale + shift), x the producer's raw fp32 NHWC output;
    fp32 NCHW [N, CO, H, W] out.  One row-streaming tensor-core kernel (dlb_head_conv_fwd)."""
    _need_cuda(x, scale, shift, w_packed, bias)
    N, H, W, Cc = x.shape
    out = torch.empty((N, CO, H, W), dtype=torch.float32, device=x.device)
    check(_lib.load().dlb_head_conv_fwd(_p(x), _p(scale), _p(shift), act, N, H, W, Cc, _p(w_packed), _p(bias), CO, border_mode,
                                        out_act, _p(out), _stream()), "dlb_head_conv_fwd")
    LAUNCHES["count"] += 1
    return out


def tile_gray_variance(img_nhwc):
    """uint8 [N,H,W,3] on device -> float64 numpy [N]: population variance of the PIL 'L' luma of every tile over its
    pixels with 0 < L < 255 (0.0 when there is none), the statistic of the reference's is_empty()."""
    _need_cuda(img_nhwc)
    N, H, W, _ = img_nhwc.shape
    sums = torch.empty((N, 3), dtype=torch.int64, device=img_nhwc.device)
    check(_lib.load().dlb_tile_luma_sums(_p(img_nhwc), N, H, W, _p(sums), _stream()), "dlb_tile_luma_sums")
    LAUNCHES["count"] += 1
    s = sums.cpu().numpy().astype("float64")
    n = s[:, 0].clip(min=1.0)
    var = s[:, 2] / n - (s[:, 1] / n) ** 2
    var[s[:, 0] == 0] = 0.0
    return var


def u8_to_f32(img_nhwc):
    _need_cuda(img_nhwc)
    N, H, W, _ = img_nhwc.shape
    out = torch.empty((N, 3, H, W), dtype=torch.float32, device=img_nhwc.device)
    check(_lib.load().dlb_u8_to_f32(_p(img_nhwc), _p(out), N, H, W, _stream()), "dlb_u8_to_f32")
    LAUNCHES["count"] += 1
    return out


def f32_to_u8(x_nchw):
    _need_cuda(x_nchw)
    N, _, H, W = x_nchw.shape
    out = torch.empty((N, H, W, 3), dtype=torch.uint8, device=x_nchw.device)
    check(_lib.load().dlb_f32_to_u8(_p(x_nchw), _p(out), N, H, W, _stream()), "dlb_f32_to_u8")
    LAUNCHES["count"] += 1
    return out


def seg_finish(segs, weights, thresh=120, want_f32=True, want_u8=True, want_mask=True, out=None):
    """segs: list of fp32 NCHW [N,3,H,W]; returns (seg_f32 NCHW, seg_u8 NHWC, mask [N,H,W]).
    out: optional (f32, u8, mask) contiguous destination tensors (e.g. batch slices) written in place."""
    _need_cuda(*segs)
    N, _, H, W = segs[0].shape
    dev = segs[0].device
    if out is not None:
        f32, u8, mask = out
        _need_cuda(f32, u8, mask)
    else:
        f32 = torch.empty((N, 3, H, W), dtype=torch.float32, device=dev) if want_f32 else None
        u8 = torch.empty((N, H, W, 3), dtype=torch.uint8, device=dev) if want_u8 else None
        mask = torch.empty((N, H, W), dtype=torch.uint8, device=dev) if want_mask else None
    ptrs = (C.c_void_p * len(segs))(*[s.data_ptr() for s in segs])
    ws = (C.c_float * len(segs))(*[float(w) for w in weights])
    check(_lib.load().dlb_seg_finish(ptrs, ws, len(segs), N, H, W, int(thresh), _p(f32), _p(u8), _p(mask), _stream()),
          "dlb_seg_finish")
    LAUNCHES["count"] += 1
    return f32, u8, mask
