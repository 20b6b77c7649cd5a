#!/usr/bin/env python
"""bench.py — 512x512 IHC tiles/sec through the five-head ResNet-9 generator path (BASELINE.json configs[1]).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the reference's CPU path (oracle port) on the host cores
    python bench.py --dump-outputs DIR ...    # also writes the last timed step's outputs (see dump_outputs)

One step = one batch of `--batch` synthetic 512x512x3 tiles through 5 ResNet-9 generators ("flat-5":
out_i = G_i(tile)), seg quantise + posneg mask.  Prints ONE JSON line (rank 0).
  value : tiles/s, inputs resident in HBM (fp32 NCHW), whole job over all ranks (weak scaling: each rank
          processes its own batch; tiles shard with no data-path collective)
  e2e   : the same through TilePipeline.infer_u8 — pinned-host uint8 tiles in, H2D, transform, generators,
          quantise, D2H of uint8 results inside the timed region
  roofline : the ResNet-block conv kernel (conv_tc, 256->256 3x3 @128x128), algorithmic FLOPs / measured
          launch time (CUDA events on the launching stream) / measured bf16 peak (MEASURED_PEAKS.json)
  cpu_baseline : oracle port (plain torch fp32 CPU, N=1 per call = reference semantics) on a bounded sample
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

HW = 512
RESNET_GFLOP = 396.41          # SURVEY.md §8d, algorithmic, per tile per generator
BLOCK_CONV_FLOP = 2 * 16384 * 256 * 2304   # one 256->256 3x3 conv @128x128, per tile
N_HEADS = 5


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=32, help="tiles per step per GPU (BASELINE configs[1]: 32)")
    ap.add_argument("--micro-batch", type=int, default=8)
    ap.add_argument("--streams", type=int, default=3, help="CUDA streams the independent generator chains are spread over")
    ap.add_argument("--precision", default="bf16x3")
    ap.add_argument("--trunk-n-tile", type=int, default=0, help="UMMA N of the ResNet-block convs (0 = 256)")
    ap.add_argument("--norm", default="batch", help="batch (CLI default of the reference) | instance")
    ap.add_argument("--workload", default="inference", choices=["inference", "train", "unet256", "cascade", "postprocess", "wsi"],
                    help="inference = BASELINE configs[1] (the headline); train = configs[3] (pix2pix step, batch 8/GPU); "
                         "unet256 = configs[4] (UNet-256 seg head, single-pass bf16, batch 64)")
    ap.add_argument("--topology", default="flat5", choices=["flat5", "default"],
                    help="train workload: flat5 = BASELINE configs[3]; default = the reference's default `deepliif train` "
                         "(4 ResNet-9 + 5 UNet-512 seg cascade, 9 n_layers=4 PatchGANs, BatchNorm, dropout, batch 1)")
    ap.add_argument("--graph", action="store_true", help="train workload: replay the step from a CUDA graph (training.GraphedStep)")
    ap.add_argument("--no-graph", action="store_true", help="inference: issue every launch from Python instead of replaying the captured CUDA graph")
    ap.add_argument("--no-extras", action="store_true", help="inference: skip the configs.{train,unet256,wsi} sub-records and the library baseline")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-roofline-events", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="inference: after the timed steps, write what the last one returned as DIR/<name>.npy (float32)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "inference" or args.impl != "b200"):
        ap.error("--dump-outputs applies to the b200 inference workload only")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", 1431.0), d.get("hbm_gbs", 6572.0), "measured"
    return 1400.0, 6650.0, "fallback"


DUMP_SAMPLE = 1 << 21          # elements kept per array: the seven outputs of a step stay under 64 MB as float32


def dump_outputs(path, outs):
    """Writes what TilePipeline.forward_device returned (four modalities, seg, seg uint8, posneg mask) as
    <path>/<name>.npy in float32.  An array of more than DUMP_SAMPLE elements is reduced to DUMP_SAMPLE of its flattened
    elements at indices drawn once from a fixed seed (sorted), so that two builds run with the same arguments can be
    compared element for element."""
    import numpy as np
    mods, seg, seg_u8, mask = outs
    arrays = {**{f"mod{i + 1}": m for i, m in enumerate(mods)}, "seg": seg, "seg_u8": seg_u8, "mask": mask}
    os.makedirs(path, exist_ok=True)
    for name, t in arrays.items():
        if t.numel() > DUMP_SAMPLE:
            idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        np.save(os.path.join(path, name + ".npy"), t.float().cpu().numpy())


# ---------------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi during the timed region)
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: oracle port on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_flat5_tiles_per_s(norm, steps, warmup):
    """Bounded sample: 1 tile x 5 ResNet-9 generators, one call per generator at N=1 (reference semantics).
    Uses the fastest torch thread count among {16, 32, 64, all cores} (probed on one generator forward each:
    oversubscribing a big host makes the N=1 oneDNN convs slower, so "all threads" is not the best it can do)."""
    from oracle import nets
    cores = os.cpu_count()
    cfg = dict(n_blocks=9, norm=norm, use_dropout=False, padding_type="zero")
    shapes = nets.resnet_param_shapes(3, 3, 64, 9, norm, False, "zero")
    sds = [nets.make_state_dict(shapes, 100 + i) for i in range(N_HEADS)]
    x = torch.rand((1, 3, HW, HW), generator=torch.Generator().manual_seed(1234)) * 2 - 1
    best_t, best_n = None, cores
    with torch.no_grad():
        for nthr in sorted({min(16, cores), min(32, cores), min(64, cores), cores}):
            torch.set_num_threads(nthr)
            nets.resnet_forward(x, sds[0], norm_mode="sample", **cfg)          # warm-up at this thread count
            t0 = time.perf_counter()
            nets.resnet_forward(x, sds[0], norm_mode="sample", **cfg)
            dt = time.perf_counter() - t0
            if best_t is None or dt < best_t:
                best_t, best_n = dt, nthr
        torch.set_num_threads(best_n)
        for _ in range(max(0, warmup - 1)):
            nets.resnet_forward(x, sds[0], norm_mode="sample", **cfg)
        t0 = time.perf_counter()
        for _ in range(steps):
            for sd in sds:
                nets.resnet_forward(x, sd, norm_mode="sample", **cfg)
        dt = time.perf_counter() - t0
    return steps / dt, dt / steps, best_n


def run_reference(args, rank):
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(1, args.warmup)
    v, s_per_step, cores = cpu_flat5_tiles_per_s(args.norm, steps, warmup)
    sample = ("1 tile (512x512x3) x 5 ResNet-9 generators per step, N=1 per call, torch fp32 CPU (oracle port), "
              "best of {16,32,64,all} threads of %d host cores" % os.cpu_count())
    line = {"impl": "reference", "metric": "512x512 IHC tiles/sec (flat-5 ResNet-9 generators)", "value": v,
            "unit": "tiles/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup,
            "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": "flat-5 ResNet-9 inference, 512x512 tiles", "norm": args.norm, "sample": sample},
            "cpu_baseline": {"value": v, "unit": "tiles/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# B200 arm
# ---------------------------------------------------------------------------------------------------
def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl b200) needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    other = {"train": bench_train, "unet256": bench_unet256, "cascade": bench_cascade, "postprocess": bench_postprocess,
             "wsi": bench_wsi}
    if args.workload in other:
        rec = other[args.workload](args, rank, world, local, dev, dist)
        if dist is not None:
            dist.barrier()
            dist.destroy_process_group()
        if rank == 0:
            print(json.dumps(rec), flush=True)
        return
    from deepliif_b200 import engine as eng_mod
    from deepliif_b200 import ops
    from deepliif_b200.models import networks
    from deepliif_b200.pipeline import TilePipeline

    # five ResNet-9 heads, random init N(0, 0.02) exactly as the reference's define_G would (no checkpoints offline)
    gens = []
    for i in range(N_HEADS):
        torch.manual_seed(i)
        g = networks.define_G(3, 3, 64, "resnet_9blocks", args.norm, args.norm == "batch", "normal", 0.02, [], "zero")
        g.precision = args.precision
        g.trunk_n_tile = args.trunk_n_tile
        g.to(dev).eval()
        gens.append(g)
    engines = [g.engine() for g in gens]
    use_graph = not args.no_graph
    pipe = TilePipeline([e.forward for e in engines], micro_batch=args.micro_batch, n_streams=args.streams, use_graph=use_graph)
    # with the graph path the first call of a shape runs eagerly (fills the caches), the second captures, later ones replay
    n_warm = max(args.warmup, 3) if use_graph else args.warmup

    B = args.batch
    # rotate over distinct input batches so the inputs of consecutive steps never sit in the 126 MB L2
    n_rot = 3
    gen = torch.Generator(device="cpu").manual_seed(1234 + rank)
    xs = [(torch.rand((B, 3, HW, HW), generator=gen) * 2 - 1).to(dev) for _ in range(n_rot)]
    u8s = [torch.randint(0, 256, (B, HW, HW, 3), dtype=torch.uint8, generator=gen).pin_memory() for _ in range(n_rot)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident metric ---------------------------------------------------------------------
    for w in range(n_warm):
        pipe.forward_device(xs[w % n_rot])
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = ops.LAUNCHES["count"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_host0 = time.perf_counter()
    for k in range(args.steps):
        outs = pipe.forward_device(xs[k % n_rot])
    t_host = time.perf_counter() - t_host0       # host enqueue time (launch-bound if close to the device time)
    e1.record()
    barrier()
    launches = ops.LAUNCHES["count"] - l0
    t_ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:          # graph replays return static buffers: read them before `pipe` runs again
        dump_outputs(args.dump_outputs, outs)
    # ---- roofline passes: the same step issued eagerly with CUDA events around every ResNet-block conv launch (events
    # cannot sit inside the replayed graph).  (a) in-region: the same stream layout as the headline, so the kernel is timed
    # while the other chains' kernels co-run; (b) isolated: ONE stream, nothing co-running ------------------------------
    roof_pairs, roof_solo = [], []
    if not args.no_roofline_events:
        for n_st, sink in ((args.streams, roof_pairs), (1, roof_solo)):
            if n_st == 1 and args.streams == 1:
                roof_solo = roof_pairs
                break
            rp = TilePipeline([e.forward for e in engines], micro_batch=args.micro_batch, n_streams=n_st)
            rp.forward_device(xs[0])
            barrier()
            eng_mod.BLOCK_CONV_EVENTS = sink
            for k in range(2):
                rp.forward_device(xs[k % n_rot])
            barrier()
            eng_mod.BLOCK_CONV_EVENTS = None
    # ---- end-to-end metric (host uint8 in, host uint8 out) ------------------------------------------------
    out_host = None
    for w in range(3 if use_graph else 1):
        out_host = pipe.infer_u8(u8s[w % n_rot], out_host)
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    for k in range(args.steps):
        out_host = pipe.infer_u8(u8s[k % n_rot], out_host)
    f1.record()
    barrier()
    clocks = sampler.stop()
    t2_ms = f0.elapsed_time(f1)
    h2d = u8s[0].numel()
    d2h = sum(v.numel() for v in out_host.values())

    tt = torch.tensor([t_ms, t2_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    t_ms, t2_ms = tt.tolist()
    tiles = B * world * args.steps
    value = tiles / (t_ms / 1e3)
    e2e = tiles / (t2_ms / 1e3)

    # ---- sub-records for the other BASELINE configs (same launch, same ranks): configs[3] training with the NCCL
    # gradient all-reduce, configs[4] UNet-256 bf16, configs[2] the WSI tile -> infer -> stitch sweep ------------------------
    extras = {}
    if not args.no_extras:
        del pipe, engines, gens, xs, u8s, out_host
        rp = None
        import gc
        gc.collect()
        torch.cuda.empty_cache()
        import copy
        for name, fn, over in (("train", bench_train, dict(batch=8, steps=3, warmup=2, graph=False, topology="flat5")),
                               ("unet256", bench_unet256, dict(batch=64, steps=10, warmup=3)),
                               ("wsi", bench_wsi, dict(steps=1, warmup=1))):
            a2 = copy.copy(args)
            for k_, v_ in over.items():
                setattr(a2, k_, v_)
            a2.no_cpu_baseline = True
            try:
                rec = fn(a2, rank, world, local, dev, dist)
            except Exception as e:                      # a failing sub-record must not lose the headline
                rec = {"error": repr(e)[:300]}
            if rank == 0 and rec is not None:
                extras[name] = _compact(rec)
            gc.collect()
            torch.cuda.empty_cache()
    if dist is not None:            # all ranks leave the group before rank 0 spends tens of seconds on the baselines
        dist.barrier()
        dist.destroy_process_group()
        dist = None

    if rank == 0:
        peak_tf, peak_hbm, peak_kind = peaks()
        whole_tf = value / world * N_HEADS * RESNET_GFLOP / 1e3            # per GPU
        roof = None

        def _kernel_rate(pairs):
            per = [a.elapsed_time(b) for a, b, _ in pairs]
            avg = sum(per) / len(per)
            return BLOCK_CONV_FLOP * pairs[0][2] / (avg * 1e-3) / 1e12, avg, len(per), pairs[0][2]
        if roof_pairs:
            ach, avg_ms, n_timed, ntile = _kernel_rate(roof_pairs)
            iso = None
            if roof_solo and roof_solo is not roof_pairs:
                a_, ms_, n_, _ = _kernel_rate(roof_solo)
                iso = {"achieved": a_, "frac": a_ / peak_tf, "launch_ms": ms_, "launches_timed": n_,
                       "note": "same kernel on ONE stream (nothing co-running)"}
            traffic = None
            tp = os.path.join(ROOT, "profiles", "block_conv_traffic.json")
            if os.path.exists(tp):
                traffic = json.load(open(tp)).get("dram_bytes_per_launch")
            roof = {"bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                    "traffic": traffic, "kernel": "conv_tc_kernel (ResNet block conv 256->256 3x3 @128x128)",
                    "launch_ms": avg_ms, "tiles_per_launch": ntile, "launches_timed": n_timed,
                    "region": "in-region: the headline step's %d-stream layout issued eagerly with CUDA events around every "
                              "block-conv launch (other chains' kernels co-run)" % args.streams,
                    "isolated": iso,
                    "whole_step_frac": whole_tf / peak_tf, "whole_step_tflops": whole_tf,
                    "peak_kind": (f"{peak_kind} cuBLAS bf16 sustained; bf16x3 executes 3 MMAs per algorithmic MAC (ceiling = 1/3)"
                                  if args.precision.endswith("x3") else peak_kind)}
        lib = None
        if not args.no_extras:
            try:
                lib = library_baseline(args, dev)
            except Exception as e:
                lib = {"error": repr(e)[:300]}
        cpu = None
        if not args.no_cpu_baseline and world == 1:          # the CPU leg is a single-GPU-run item (rank 0, N=1 only)
            v, s_per, cores = cpu_flat5_tiles_per_s(args.norm, 1, 1)
            cpu = {"value": v, "unit": "tiles/s", "cores": cores, "kind": "port",
                   "sample": "1 tile x 5 ResNet-9 generators, N=1 per call, torch fp32 CPU (oracle port), best of {16,32,64,all} threads, 1 warm-up", "host_cores": os.cpu_count()}
        line = {
            "metric": "512x512 IHC tiles/sec (flat-5 ResNet-9 generators)", "value": value, "unit": "tiles/s",
            "n_gpus": world, "steps": args.steps, "warmup": n_warm, "ms_per_step": t_ms / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32 result via %s tensor-core operands, fp32 accumulate" % args.precision, "data": "synthetic",
            "config": {"workload": "inference: 5x ResNet-9blocks generators, batch=%d/GPU, 512x512 synthetic tiles"
                                   % B, "norm": args.norm, "padding": "zero", "micro_batch": args.micro_batch, "streams": args.streams,
                       "cuda_graph": use_graph,
                       "fused_operand": {k: os.environ.get(k, "default") for k in ("DLB_FUSED", "DLB_FUSE_RESIDUAL", "DLB_FUSE_STEM",
                                                                                      "DLB_FUSE_UP", "DLB_FUSE_HEAD", "DLB_STEM_STREAM",
                                                                                      "DLB_HEAD_STREAM", "DLB_EPI_SMEM", "DLB_EPI2", "DLB_CTA2")},
                       "host_enqueue_ms_per_step": t_host * 1e3 / args.steps,
                       "parallelism": "tile-sharded dp%d, no collective" % world,
                       "l2": "3 rotating input batches (%.0f MB each) + multi-GB activations per step >> 126 MB L2" % (B * 3 * HW * HW * 4 / 1e6),
                       "algorithmic_gflop_per_tile": N_HEADS * RESNET_GFLOP},
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "tiles/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "ms_per_step": t2_ms / args.steps},
            "gpu_launches": launches,
            "roofline": roof, "cpu_baseline": cpu, "library_baseline": lib,
            "algorithmic_tflops": value * N_HEADS * RESNET_GFLOP / 1e3,
            "configs": extras or None,
        }
        print(json.dumps(line), flush=True)


def _compact(rec):
    """Sub-record of the headline line: the numbers, not the prose."""
    if rec is None or "error" in rec:
        return rec
    keep = ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "dtype", "gpu_launches",
            "algorithmic_tflops", "e2e", "roofline", "cuda_graph", "sweep", "loss_G_L1_1")
    out = {k: rec[k] for k in keep if k in rec}
    out["workload"] = rec.get("config", {}).get("workload")
    for k in ("host_enqueue_ms_per_step", "parallelism", "allreduce"):
        if k in rec.get("config", {}):
            out[k] = rec["config"][k]
    return out


def library_baseline(args, dev):
    """The "library bar" (SURVEY.md 8d): the same five ResNet-9 generators as plain torch.nn.functional calls on THIS GPU —
    eager PyTorch over cuDNN, which is what the reference's modules execute (networks.py:448-450) — batch 32, fp32 inputs
    resident in HBM, (a) with TF32 convolutions allowed (the reference default, cli.py:1059-1063) and (b) strict fp32.
    Also reports each variant's max-abs error against the CPU fp32 oracle on one tile (the 1e-3 parity gate)."""
    from oracle import nets
    cfg = dict(n_blocks=9, norm=args.norm, use_dropout=False, padding_type="zero")
    shapes = nets.resnet_param_shapes(3, 3, 64, 9, args.norm, False, "zero")
    sds_cpu = [nets.make_state_dict(shapes, 100 + i) for i in range(N_HEADS)]
    sds = [{k: v.to(dev) for k, v in sd.items()} for sd in sds_cpu]
    B = args.batch
    g = torch.Generator().manual_seed(77)
    x_cpu = torch.rand((B, 3, HW, HW), generator=g) * 2 - 1
    x = x_cpu.to(dev)
    with torch.no_grad():
        torch.set_num_threads(min(32, os.cpu_count()))
        y_ref = nets.resnet_forward(x_cpu[:1], sds_cpu[0], norm_mode="sample", **cfg)
    out = {"what": "oracle/nets.resnet_forward on cuda (eager PyTorch, cuDNN convolutions, F.instance_norm), 5 generators, "
                   "batch %d in micro-batches of %d, device-resident fp32 input" % (B, args.micro_batch), "unit": "tiles/s"}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        torch.backends.cudnn.benchmark = True
        for label, tf32 in (("tf32", True), ("fp32", False)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32

            def step():
                with torch.no_grad():
                    for sd in sds:
                        for s0 in range(0, B, args.micro_batch):
                            nets.resnet_forward(x[s0:s0 + args.micro_batch], sd, norm_mode="sample", **cfg)
            step(); step()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(2):
                step()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 2
            with torch.no_grad():
                y = nets.resnet_forward(x[:1], sds[0], norm_mode="sample", **cfg).cpu()
            err = float((y - y_ref).abs().max())
            out[label] = {"value": B / (ms / 1e3), "ms_per_step": ms, "max_abs_vs_cpu_oracle": err, "passes_1e-3": err <= 1e-3}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    return out


# ROI sizes (W, H) of the reference's Sample_Large_Tissues/ PNGs (the images themselves cannot travel to the GPU box)
WSI_ROIS = [(1381, 949), (1404, 1179), (2167, 1520), (2662, 2207), (1250, 995)]


def bench_wsi(args, rank, world, local, dev, dist):
    """BASELINE configs[2]: the WSI sweep — five Sample_Large_Tissues-sized ROIs through models.infer_tiles (the body of
    inference(), models/__init__.py:464-579): InferenceTiler geometry at tile_size=512 overlap=56 (102 tiles), tiles sharded
    rank::world, the default cascade (4 ResNet-9 + 5 UNet-512) on every rank, uint8 results gathered to rank 0 (one NCCL
    gather per ROI) and stitched there.  Timed end to end with the host work inside (tiling, pinning, H2D, D2H, gather,
    stitching): wall clock between barriers, max over ranks."""
    import numpy as np
    from PIL import Image
    from deepliif_b200 import ops
    from deepliif_b200.models import infer_tiles, networks
    from deepliif_b200.options import Options
    opt = Options(d_params=dict(model="DeepLIIF", name="bench", checkpoints_dir="/tmp", gpu_ids=(local,), input_nc=3, output_nc=3,
                                ngf=64, ndf=64, net_g="resnet_9blocks", net_gs="unet_512", net_d="n_layers", norm=args.norm,
                                no_dropout=False, padding="zero", init_type="normal", init_gain=0.02, modalities_no=4, seg_gen=True,
                                input_no=1, scale_size=512, phase="test", modalities_names=["IHC", "Hema", "DAPI", "Lap2", "Marker"],
                                seg_weights=[0.25, 0.15, 0.25, 0.1, 0.25], loss_G_weights=[0.2] * 5, loss_D_weights=[0.2] * 5,
                                mod_id_seg="S", background_colors=[[255, 255, 255]] * 4), mode="train")
    opt.input_id = "0"
    nets = {}
    for i in range(1, 5):
        torch.manual_seed(i)
        nets[f"G{i}"] = networks.define_G(3, 3, 64, "resnet_9blocks", args.norm, True, "normal", 0.02, [], "zero").to(dev).eval()
    for i in range(5):
        torch.manual_seed(10 + i)
        nets[f"GS{i}"] = networks.define_G(3, 3, 64, "unet_512", args.norm, True, "normal", 0.02, []).to(dev).eval()
    rng = np.random.default_rng(7)          # same images on every rank
    rois = []
    for (W_, H_) in WSI_ROIS:
        small = rng.integers(0, 256, size=(H_ // 8 + 2, W_ // 8 + 2, 3)).astype(np.float32)
        img = np.kron(small, np.ones((8, 8, 1), np.float32))[:H_, :W_]
        img = 0.75 * img + 0.25 * rng.integers(0, 256, size=(H_, W_, 3)).astype(np.float32)
        rois.append(Image.fromarray(np.clip(img, 0, 255).astype(np.uint8)))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    from deepliif_b200.util import TileGrid
    tiles_per_sweep = sum(len(TileGrid(np.asarray(im), 512, 56).tiles()) for im in rois)

    from deepliif_b200.models import infer_images

    def sweep():
        outs = None
        # what inference() runs by default: the four modalities + Seg (no per-modality seg intermediates); the five ROIs go
        # through the pipelined per-image loop (tiling / upload of ROI k+1 and stitching of ROI k-1 overlap the GPU work of k)
        for _, res in infer_images(rois, 512, 56, nets, opt, seg_weights=opt.seg_weights, want_parts=False):
            outs = res if res is not None else outs
        return (tiles_per_sweep if rank == 0 else 0), outs

    for _ in range(max(1, args.warmup) + 1):     # first sweep: eager (fills caches); second: captures the per-shape graphs
        sweep()
    barrier()
    l0 = ops.LAUNCHES["count"]
    sampler = ClockSampler(local); sampler.start()
    t0 = time.perf_counter()
    n_tiles = 0
    for _ in range(args.steps):
        n, outs = sweep()
        n_tiles += n
    barrier()
    dt = time.perf_counter() - t0
    clocks = sampler.stop()
    t = torch.tensor([dt], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dt = float(t.item())
    if rank == 0:
        v = n_tiles / dt
        return {"metric": "WSI sweep tiles/sec (5 ROIs, tile 512 overlap 56, default cascade), end to end incl. tiling + stitch", "value": v,
                "unit": "tiles/s", "n_gpus": world, "steps": args.steps, "warmup": max(1, args.warmup) + 1, "ms_per_step": dt * 1e3 / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32 via %s" % args.precision,
                "data": "synthetic", "config": {"workload": "WSI sweep: 5 ROIs sized like Sample_Large_Tissues (%s), tile_size=512 "
                                                            "overlap=56 -> %d tiles per sweep, tiles sharded over %d GPU(s), rank-0 stitch"
                                                            % (", ".join("%dx%d" % r for r in WSI_ROIS), n_tiles // max(1, args.steps), world),
                                                "norm": args.norm, "parallelism": "tile-sharded dp%d + 1 gather per ROI, host tiling / stitching pipelined across ROIs" % world},
                "clocks": clocks, "gpu_launches": ops.LAUNCHES["count"] - l0,
                "sweep": {"seconds": dt / args.steps, "tiles": n_tiles // max(1, args.steps), "rois": len(rois),
                          "outputs_per_roi": sorted(outs.keys()) if outs else None},
                "e2e": {"value": v, "unit": "tiles/s",
                        "h2d_bytes_per_step": n_tiles // max(1, args.steps) * 512 * 512 * 3,
                        "d2h_bytes_per_step": n_tiles // max(1, args.steps) * 512 * 512 * 3 * 5}}
    return None


def bench_cascade(args, rank, world, local, dev, dist):
    """The reference's default `deepliif test` topology: 4 ResNet-9 modality generators + 5 UNet-512 seg generators in
    cascade (DeepLIIF_model.py:175-203; 1827.8 GFLOP/tile), end to end from pinned-host uint8 tiles to uint8 results."""
    from deepliif_b200 import ops
    from deepliif_b200.models import networks
    from deepliif_b200.pipeline import TilePipeline
    B = args.batch
    gens, segs = [], []
    for i in range(4):
        torch.manual_seed(i)
        gens.append(networks.define_G(3, 3, 64, "resnet_9blocks", args.norm, True, "normal", 0.02, [], "zero").to(dev).eval())
    for i in range(5):
        torch.manual_seed(10 + i)
        segs.append(networks.define_G(3, 3, 64, "unet_512", args.norm, True, "normal", 0.02, []).to(dev).eval())
    pipe = TilePipeline([g.engine().forward for g in gens], [s_.engine().forward for s_ in segs], [0.25, 0.15, 0.25, 0.1, 0.25],
                        micro_batch=args.micro_batch, n_streams=args.streams)
    gen = torch.Generator().manual_seed(99 + rank)
    u8s = [torch.randint(0, 256, (B, HW, HW, 3), dtype=torch.uint8, generator=gen).pin_memory() for _ in range(3)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    out = None
    for w in range(args.warmup):
        out = pipe.infer_u8(u8s[w % 3], out)
    barrier()
    sampler = ClockSampler(local); sampler.start()
    l0 = ops.LAUNCHES["count"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        out = pipe.infer_u8(u8s[k % 3], out)
    e1.record()
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_ms = float(t.item())
    if rank == 0:
        v = B * world * args.steps / (t_ms / 1e3)
        return ({"metric": "512x512 IHC tiles/sec (default cascade: 4 ResNet-9 + 5 UNet-512), end to end", "value": v,
                          "unit": "tiles/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32 via %s" % args.precision, "data": "synthetic",
                          "config": {"workload": "inference: DeepLIIF default cascade, batch=%d/GPU, host uint8 in/out" % B,
                                     "norm": args.norm, "micro_batch": args.micro_batch, "streams": args.streams},
                          "clocks": clocks, "gpu_launches": ops.LAUNCHES["count"] - l0,
                          "algorithmic_tflops": v * 1827.8 / 1e3})
    return None


def bench_postprocess(args, rank, world, local, dev, dist):
    """SURVEY 8(f) row 2: compute_final_results (postprocessing.py:1223-1304) on one stitched region — create_posneg_mask,
    mark_background, cell labelling + statistics, classification, boundary growth, overlay / refined images.  Each rank
    processes its own region (regions are independent: no collective)."""
    import numpy as np
    from oracle import cells as C                          # input synthesis + the cpu_baseline leg only
    from deepliif_b200 import ops
    from deepliif_b200 import postprocessing as P
    T, REP = 2048, 4
    o, s_, m = C.synth_case(T, T, 500 + rank)
    orig, seg, marker = (np.ascontiguousarray(np.tile(a, (REP, REP, 1))) for a in (o, s_, m))
    H, W = orig.shape[:2]
    kw = dict(marker_thresh="default", large_noise_thresh="default")
    d_in = [torch.from_numpy(a).to(dev) for a in (orig, seg, marker)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local); sampler.start()
    l0 = ops.LAUNCHES["count"]
    t_dev = timed(lambda: P.compute_final_results_device(d_in[0], d_in[1], d_in[2], "40x", **kw))
    launches = (ops.LAUNCHES["count"] - l0) // (args.steps + args.warmup) * args.steps
    clocks = sampler.stop()

    t_e2e = timed(lambda: P.compute_final_results(orig, seg, marker, "40x", **kw))     # the public call: numpy in, numpy out
    clock = P.StageClock()
    _, _, scoring, _, cells = P.compute_final_results_device(d_in[0], d_in[1], d_in[2], "40x", clock=clock, **kw)
    stages = clock.ms()
    if rank == 0:
        mp = H * W / 1e6
        v = mp * world * args.steps / (t_dev / 1e3)
        pk = peaks()
        alg_bytes = 15.0 * H * W                           # 3 uint8 images read, 2 written: the floor for this function
        dev_ms = sum(v_ for k, v_ in stages.items() if k != "host thresholds")
        line = {"metric": "stitched-region cell post-processing (compute_final_results), Mpixel/s", "value": v, "unit": "Mpixel/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_dev / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8 / int32", "data": "synthetic",
                "config": {"workload": "postprocess: %dx%d region (%dx%d synthetic tile repeated %dx%d), %d cells, 40x defaults"
                                       % (H, W, T, T, REP, REP, len(cells)),
                           "l2": "per-step working set %.0f MB >> 126 MB L2" % (H * W * 25 / 1e6)},
                "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": mp * world * args.steps / (t_e2e / 1e3), "unit": "Mpixel/s", "h2d_bytes_per_step": 9 * H * W,
                        "d2h_bytes_per_step": 6 * H * W},
                "stages_ms": stages,
                "roofline": {"bound": "hbm", "achieved": alg_bytes / (dev_ms / 1e3) / 1e9, "peak": pk[1], "unit": "GB/s",
                             "frac": alg_bytes / (dev_ms / 1e3) / 1e9 / pk[1], "peak_source": pk[2], "traffic": None,
                             "note": "whole device pipeline (all kernels of the function; host threshold step excluded); "
                                     "algorithmic bytes = 15 B/pixel"}}
        if not args.no_cpu_baseline and world == 1:
            t0 = time.perf_counter()
            C.compute_final_results(o, s_, m, "40x", **kw)
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": T * T / 1e6 / dt, "unit": "Mpixel/s", "cores": 1, "kind": "port",
                                    "sample": "one %dx%d tile of the region through oracle/cells.py (numpy/scipy)" % (T, T)}
        return line
    return None


def bench_unet256(args, rank, world, local, dev, dist):
    """BASELINE configs[4]: UNet-256 generator (8 downs), single-pass bf16 operands, batch 64, seg head only,
    256x256 tiles (bottleneck 1x1).  Exercises the ConvTranspose2d path (4-phase tcgen05 GEMMs, dual-source skip)."""
    from deepliif_b200 import ops
    from deepliif_b200.models import networks
    from deepliif_b200.pipeline import TilePipeline
    B = 64 if args.batch == 32 else args.batch
    prec = "bf16" if args.precision == "bf16x3" else args.precision
    torch.manual_seed(0)
    net = networks.define_G(3, 3, 64, "unet_256", args.norm, False, "normal", 0.02, [])
    net.precision = prec
    net.to(dev).eval()
    eng = net.engine()
    pipe = TilePipeline([eng.forward], micro_batch=B, n_streams=1)
    g = torch.Generator().manual_seed(4321 + rank)
    xs = [(torch.rand((B, 3, 256, 256), generator=g) * 2 - 1).to(dev) for _ in range(3)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for w in range(args.warmup):
        pipe.forward_device(xs[w % 3])
    barrier()
    # The ~90 launches of this small network are launch-bound from Python: replay them from a CUDA graph.
    graph, static_x = None, xs[0].clone()
    try:
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            pipe.forward_device(static_x)
        torch.cuda.current_stream().wait_stream(side)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            static_out = pipe.forward_device(static_x)
    except Exception as e:      # capture is an optimisation only
        graph = None
        print("cuda graph capture failed, running eagerly:", repr(e)[:200], file=sys.stderr)
    launches_per_step = None

    def step(k):
        if graph is not None:
            static_x.copy_(xs[k % 3]); graph.replay()
        else:
            pipe.forward_device(xs[k % 3])

    for w in range(3):
        step(w)
    barrier()
    sampler = ClockSampler(local); sampler.start()
    l0 = ops.LAUNCHES["count"]
    pipe_l0 = l0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        step(k)
    e1.record()
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_ms = float(t.item())
    if graph is not None:       # launches replayed by the graph are not seen by the Python counter: count one eager pass
        c0 = ops.LAUNCHES["count"]; pipe.forward_device(xs[0]); torch.cuda.synchronize()
        ops.LAUNCHES["count"] = l0 + (ops.LAUNCHES["count"] - c0) * args.steps
    if rank == 0:
        v = B * world * args.steps / (t_ms / 1e3)
        pk = peaks()
        return ({"metric": "256x256 tiles/sec (UNet-256 seg head)", "cuda_graph": graph is not None, "value": v, "unit": "tiles/s", "n_gpus": world,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": t_ms / args.steps, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": prec, "data": "synthetic",
                          "config": {"workload": "UNet-256 generator, %s, batch=%d/GPU, seg head only, 256x256" % (prec, B),
                                     "norm": args.norm}, "clocks": clocks, "gpu_launches": ops.LAUNCHES["count"] - l0,
                          "algorithmic_tflops": v * 12.10 / 1e3,
                          "roofline": {"bound": "tensor", "achieved": v / world * 12.10 / 1e3, "peak": pk[0], "unit": "TFLOP/s",
                                       "frac": v / world * 12.10 / 1e3 / pk[0], "traffic": None,
                                       "note": "whole network (single-pass bf16: ceiling 1.0), algorithmic 12.10 GFLOP/tile"}})
    return None


def bench_train(args, rank, world, local, dev, dist):
    """BASELINE configs[3]: pix2pix L1+GAN step, 5x (ResNet-9 G + 70x70 PatchGAN D), batch 8/GPU, flat-bucket
    all-reduce.  One step = DeepLIIFModel.optimize_parameters() on a synthetic batch resident in HBM."""
    from deepliif_b200 import ops, training
    from deepliif_b200.cli import TRAIN_DEFAULTS
    from deepliif_b200.models import create_model
    default_topo = args.topology == "default"
    B = (1 if default_topo else 8) if args.batch == 32 else args.batch
    if default_topo:
        p = dict(TRAIN_DEFAULTS, dataroot="/tmp", checkpoints_dir="/tmp/dlb_bench_ckpt", name="bench", gpu_ids=(local,),
                 batch_size=B, precision=args.precision)          # everything else = the CLI defaults
    else:
        p = dict(TRAIN_DEFAULTS, dataroot="/tmp", checkpoints_dir="/tmp/dlb_bench_ckpt", name="bench", gpu_ids=(local,),
                 modalities_no=N_HEADS, seg_gen=False, norm="instance", no_dropout=True, padding="zero", net_g="resnet_9blocks",
                 net_d="basic", batch_size=B, precision=args.precision)
    opt = training.build_options(p)
    torch.manual_seed(0)
    model = create_model(opt)
    training.make_optimizers(model)
    model.train()
    g = torch.Generator().manual_seed(100 + rank)
    batches = [{"A": (torch.rand((B, 3, HW, HW), generator=g) * 2 - 1).to(dev),
                "B": [(torch.rand((B, 3, HW, HW), generator=g) * 2 - 1).to(dev) for _ in range(5 if default_topo else N_HEADS)],
                "A_paths": []}
               for _ in range(2)]

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    stepper = training.GraphedStep(model, warmup=2) if args.graph else None

    def one_step(k):
        if stepper is not None:
            stepper(batches[k % 2])
        else:
            model.set_input(batches[k % 2]); model.optimize_parameters()

    per_step_launches = 0
    for w in range(max(args.warmup, 3) if stepper is not None else args.warmup):
        c0 = ops.LAUNCHES["count"]
        one_step(w)
        if w == 0:
            per_step_launches = ops.LAUNCHES["count"] - c0      # an eager step: what one graph replay re-issues
    barrier()
    sampler = ClockSampler(local); sampler.start()
    l0 = ops.LAUNCHES["count"]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    t_h0 = time.perf_counter()
    for k in range(args.steps):
        one_step(k)
    t_host = time.perf_counter() - t_h0
    e1.record()
    barrier()
    clocks = sampler.stop()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    t_ms = float(t.item())
    if rank == 0:
        losses = model.get_current_losses()
        # algorithmic FLOPs per tile: G fwd + bwd (2x) for 5 heads, D: 3 fwd + 2 bwd(params) + 1 bwd(data) per head
        gflop = (N_HEADS * (3 * RESNET_GFLOP + (3 + 2 * 2 + 1) * 26.11) if not default_topo else
                 3 * (4 * RESNET_GFLOP + 5 * 48.44) + 9 * (3 + 2 * 2 + 1) * 21.77)
        v = B * world * args.steps / (t_ms / 1e3)
        return ({"metric": ("512x512 training tiles/sec (DeepLIIF default step: 4 ResNet-9 + 5 UNet-512 G, 9 PatchGAN D)"
                                     if default_topo else
                                     "512x512 training tiles/sec (pix2pix step, 5x ResNet-9 G + PatchGAN D)"), "value": v,
                          "unit": "tiles/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": t_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                          "dtype": "f32 via %s tensor-core operands" % args.precision, "data": "synthetic",
                          "config": {"workload": ("training: reference default topology (4 ResNet-9 + 5 UNet-512 cascade, 9 PatchGAN "
                                                  "n_layers=4, BatchNorm, dropout), batch=%d/GPU" % B) if default_topo else
                                                 ("training: pix2pix L1+GAN, 5x (ResNet-9blocks G + 70x70 PatchGAN D), "
                                                  "batch=%d/GPU, flat-bucket all-reduce" % B), "norm": opt.norm,
                                     "parallelism": "dp%d" % world, "host_enqueue_ms_per_step": t_host * 1e3 / args.steps,
                                     "cuda_graph": stepper is not None},
                          "clocks": clocks,
                          "gpu_launches": per_step_launches * args.steps if stepper is not None else ops.LAUNCHES["count"] - l0,
                          "algorithmic_tflops": v * gflop / 1e3, "loss_G_L1_1": losses.get("G_L1_1")})
    return None


if __name__ == "__main__":
    main()
