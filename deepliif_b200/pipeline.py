"""Tile-batched inference driver: uint8 tiles in (host) -> five uint8 outputs + posneg mask out (host).

Replaces the reference's per-tile loop ``inference -> run_wrapper -> run_dask`` (deepliif/models/__init__.py:
464-579, 258-361), which runs batch = 1 and converts PIL <-> tensor <-> PIL around every generator call, with a
batched device pipeline: one H2D copy of the uint8 tiles, on-GPU ``transform`` (data/__init__.py:133-138), the
generators in micro-batches sized for L2 residency, on-GPU ``tensor2im`` quantisation (util/util.py:130-135),
seg aggregation + ``create_posneg_mask`` (models/__init__.py:338, postprocessing.py:163-190), one D2H copy of
uint8 results.  Two graph shapes:

  flat     : out_i = G_i(x), i = 1..5 (BASELINE.json configs 1-2: five ResNet-9 heads on the IHC tile; the
             fifth is the Seg head)
  cascade  : mods_i = G_i(x) (i = 1..4); seg = sum_k w_k * GS_k(x | mods_k)   (DeepLIIF_model.py:175-203)
             Entries of `gens` / `segs` may be None: that branch is pruned (``seg_only`` with zero seg weights,
             models/__init__.py:318-319) — a pruned modality generator needs its seg generator pruned too.

Launch path.  A step is ~1250 kernel launches; issued one by one from Python they cost more host time than the GPU
needs to run them.  With ``use_graph`` the whole step for a given batch shape (all streams, all micro-batches) is
captured ONCE into a CUDA graph (every launch goes through the same C-ABI calls while the stream is capturing:
tensor maps are encoded and activation buffers taken from the graph's private pool at capture time only) and a step
is then one ``cudaGraphLaunch`` on static input / output buffers.
"""
import torch

from . import ops


class _Captured:
    __slots__ = ("graph", "static_in", "outs", "launches", "engines")


class TilePipeline:
    def __init__(self, gens, segs=None, seg_weights=None, micro_batch=8, thresh=120, n_streams=3, use_graph=False):
        """gens: list of callables fp32 NCHW -> fp32 NCHW (modalities).  segs: None (flat: last of `gens` is the
        seg head) or list of len(gens)+1 seg generators (cascade)."""
        self.gens, self.segs = list(gens), (list(segs) if segs is not None else None)
        n_seg = len(self.segs) if self.segs is not None else 1
        self.seg_weights = list(seg_weights) if seg_weights is not None else [1.0 / n_seg] * n_seg
        if self.segs is not None:
            assert len(self.segs) == len(self.gens) + 1, "cascade: one seg generator per modality + the base one"
            for i, g in enumerate(self.gens):
                assert g is not None or self.segs[i + 1] is None, "a pruned modality generator cannot feed a seg generator"
            assert any(s is not None for s in self.segs), "cascade: every seg generator is pruned"
        self.micro_batch, self.thresh = micro_batch, thresh
        self.n_streams, self._stream_cache = n_streams, {}
        self.use_graph = use_graph
        self._graphs, self._seen = {}, set()
        self._keep_parts = None
        # positions of `gens` whose outputs are modalities (returned in this order by forward_device / infer_u8)
        n_mod = len(self.gens) - (1 if self.segs is None else 0)
        self.mod_index = [i for i in range(n_mod) if self.gens[i] is not None]
        self.part_index = [k for k, s in enumerate(self.segs) if s is not None] if self.segs is not None else []

    # ---- the step itself (eager issue; also what a graph capture records) -------------------------------------------
    @torch.no_grad()
    def _forward_eager(self, x):
        N, _, H, W = x.shape
        dev = x.device
        mb = self.micro_batch if self.micro_batch > 0 else N
        mods_out = {i: torch.empty((N, 3, H, W), dtype=torch.float32, device=dev) for i in self.mod_index}
        seg_out = torch.empty((N, 3, H, W), dtype=torch.float32, device=dev)
        segu8_out = torch.empty((N, H, W, 3), dtype=torch.uint8, device=dev)
        mask_out = torch.empty((N, H, W), dtype=torch.uint8, device=dev)
        keep_parts = self._keep_parts is not None and self.segs is not None
        self._parts_out = ({k: torch.empty((N, 3, H, W), dtype=torch.float32, device=dev) for k in self.part_index}
                           if keep_parts else None)
        main = torch.cuda.current_stream()
        streams = self._streams(dev)
        for st in streams:
            st.wait_stream(main)
        k = 0
        for s in range(0, N, mb):
            xs = x[s:s + mb]
            if self.segs is None:
                n_mod = len(self.gens) - 1
                for i, g in enumerate(self.gens):
                    st = streams[k % len(streams)]; k += 1
                    with torch.cuda.stream(st):
                        o = g(xs)
                        if i < n_mod:
                            mods_out[i][s:s + mb].copy_(o)
                        else:
                            ops.seg_finish([o], [1.0], self.thresh, out=(seg_out[s:s + mb], segu8_out[s:s + mb], mask_out[s:s + mb]))
            else:
                # cascade: modality chain i feeds seg generator i+1; the base seg generator reads the tile itself
                parts, wts = [], []
                used = []
                for i in range(len(self.segs)):
                    gen = self.gens[i - 1] if i > 0 else None
                    if self.segs[i] is None and gen is None:
                        continue
                    st = streams[k % len(streams)]; k += 1
                    used.append(st)
                    with torch.cuda.stream(st):
                        src = xs
                        if i > 0:
                            src = gen(xs)
                            mods_out[i - 1][s:s + mb].copy_(src)
                        if self.segs[i] is not None:
                            p = self.segs[i](src)
                            parts.append(p); wts.append(self.seg_weights[i])
                            if keep_parts:
                                self._parts_out[i][s:s + mb].copy_(p)
                fin = used[0]
                for st in used[1:]:
                    fin.wait_stream(st)
                with torch.cuda.stream(fin):
                    ops.seg_finish(parts, wts, self.thresh, out=(seg_out[s:s + mb], segu8_out[s:s + mb], mask_out[s:s + mb]))
                for st in used[1:]:
                    st.wait_stream(fin)      # parts stay alive until seg_finish has consumed them
        for st in streams:
            main.wait_stream(st)
        return [mods_out[i] for i in self.mod_index], seg_out, segu8_out, mask_out

    def _streams(self, dev):
        if self.n_streams <= 1:
            return [torch.cuda.current_stream()]
        key = str(dev)
        if key not in self._stream_cache:
            self._stream_cache[key] = [torch.cuda.Stream(device=dev) for _ in range(self.n_streams)]
        return self._stream_cache[key]

    # ---- CUDA-graph replay ----------------------------------------------------------------------------------------------
    def _engines(self):
        """The engine every network runs with now.  net.engine() rebuilds it when the network's weights or precision
        changed, so a replay can tell whether its graph still matches the networks.  None for a plain callable."""
        return [n.engine() if hasattr(n, "engine") else None for n in self.gens + (self.segs or []) if n is not None]

    def _graphed(self, kind, shape, dtype, dev, body):
        """Captured graph of `body(static_in)` for this input shape, or None the first time the shape is seen (the
        caller then runs eagerly, which doubles as the warm-up that fills the workspace caches).  A graph bakes in the
        engines' weight buffers: once any network has rebuilt its engine, every graph is dropped and the shape starts
        over (eager, then captured again)."""
        key = (kind, tuple(shape), dtype, str(dev), self._keep_parts is not None)
        cap = self._graphs.get(key)
        if cap is not None:
            if all(a is b for a, b in zip(self._engines(), cap.engines)):
                return cap
            torch.cuda.synchronize()      # a replay still in flight reads the graph pool and the old weights
            self._graphs.clear()
            self._seen.clear()
        if key not in self._seen:
            self._seen.add(key)
            return None
        cap = _Captured()
        cap.static_in = torch.zeros(tuple(shape), dtype=dtype, device=dev)
        cap.engines = self._engines()
        torch.cuda.synchronize()
        l0 = ops.LAUNCHES["count"]
        cap.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(cap.graph):
            cap.outs = body(cap.static_in)
        cap.launches = ops.LAUNCHES["count"] - l0
        ops.LAUNCHES["count"] = l0
        self._graphs[key] = cap
        return cap

    @torch.no_grad()
    def forward_device(self, x):
        """x: fp32 NCHW on device.  Returns (list of modality fp32 NCHW, seg fp32 NCHW, seg_u8 NHWC, mask).

        Independent (micro-batch, generator) chains are issued round-robin on `n_streams` CUDA streams: the
        memory-bound passes of one chain (normalise/split, statistics) then overlap the tensor-core-bound
        convolutions of another, and wave-quantisation tails are filled.  With use_graph the outputs are the
        graph's static buffers: consume them before the next call with the same shape."""
        if not self.use_graph:
            return self._forward_eager(x)
        cap = self._graphed("dev", x.shape, x.dtype, x.device, self._forward_eager)
        if cap is None:
            return self._forward_eager(x)
        cap.static_in.copy_(x)
        cap.graph.replay()
        ops.LAUNCHES["count"] += cap.launches
        return cap.outs

    def _u8_body(self, x_u8):
        x = ops.u8_to_f32(x_u8)
        mods, seg, seg_u8, mask = self._forward_eager(x)
        dev = x.device
        mods_u8 = torch.stack([ops.f32_to_u8(m) for m in mods]) if mods else torch.empty((0,) + tuple(seg_u8.shape),
                                                                                          dtype=torch.uint8, device=dev)
        parts_u8 = None
        if self._keep_parts is not None and self._parts_out is not None:
            parts_u8 = torch.stack([ops.f32_to_u8(self._parts_out[k]) for k in self.part_index])
        return mods_u8, seg_u8, mask, parts_u8

    @torch.no_grad()
    def infer_u8(self, tiles_u8_host, out_host=None, want_parts=False):
        """tiles_u8_host: pinned uint8 [N,H,W,3].  Returns dict of pinned uint8 host tensors:
        'mods' [M,N,H,W,3], 'seg' [N,H,W,3], 'mask' [N,H,W] (+ 'parts' [K,N,H,W,3], the per-modality seg outputs,
        when want_parts).  Copies are part of the call (end-to-end path); the D2H copies are asynchronous on the
        current stream — synchronise before reading."""
        dev = torch.device("cuda", torch.cuda.current_device())
        self._keep_parts = [] if want_parts else None
        cap = None
        if self.use_graph:
            cap = self._graphed("u8", tiles_u8_host.shape, torch.uint8, dev, self._u8_body)
        if cap is not None:
            cap.static_in.copy_(tiles_u8_host, non_blocking=True)
            cap.graph.replay()
            ops.LAUNCHES["count"] += cap.launches
            mods_u8, seg_u8, mask, parts_u8 = cap.outs
        else:
            x_u8 = tiles_u8_host.to(dev, non_blocking=True)
            mods_u8, seg_u8, mask, parts_u8 = self._u8_body(x_u8)
        if out_host is None:
            out_host = {"mods": torch.empty(mods_u8.shape, dtype=torch.uint8, pin_memory=True),
                        "seg": torch.empty(seg_u8.shape, dtype=torch.uint8, pin_memory=True),
                        "mask": torch.empty(mask.shape, dtype=torch.uint8, pin_memory=True)}
        out_host["mods"].copy_(mods_u8, non_blocking=True)
        out_host["seg"].copy_(seg_u8, non_blocking=True)
        out_host["mask"].copy_(mask, non_blocking=True)
        if want_parts:
            if "parts" not in out_host:
                out_host["parts"] = torch.empty(parts_u8.shape, dtype=torch.uint8, pin_memory=True)
            out_host["parts"].copy_(parts_u8, non_blocking=True)
        return out_host

    @torch.no_grad()
    def infer_u8_device(self, x_u8, want_parts=False):
        """x_u8: uint8 [N,H,W,3] already on the device.  Returns device tensors (mods_u8 [M,N,H,W,3], seg_u8 [N,H,W,3],
        mask [N,H,W], parts_u8 [K,N,H,W,3] | None).  With use_graph these are the captured graph's static buffers: consume
        (copy / scatter) them before the next call of the same shape."""
        self._keep_parts = [] if want_parts else None
        cap = None
        if self.use_graph:
            cap = self._graphed("u8", x_u8.shape, torch.uint8, x_u8.device, self._u8_body)
        if cap is not None:
            cap.static_in.copy_(x_u8, non_blocking=True)
            cap.graph.replay()
            ops.LAUNCHES["count"] += cap.launches
            return cap.outs
        return self._u8_body(x_u8.contiguous())

    @torch.no_grad()
    def infer_mods_u8(self, tiles_u8_host):
        """Modalities only (mod_only / seg_gen=False): no seg generators are run."""
        dev = torch.device("cuda", torch.cuda.current_device())
        x = ops.u8_to_f32(tiles_u8_host.to(dev, non_blocking=True))
        mb = self.micro_batch if self.micro_batch > 0 else x.shape[0]
        gens = [self.gens[i] for i in self.mod_index] if self.segs is not None else [g for g in self.gens if g is not None]
        outs = [torch.cat([g(x[s:s + mb]) for s in range(0, x.shape[0], mb)]) for g in gens]
        mods_u8 = torch.stack([ops.f32_to_u8(m) for m in outs])
        host = torch.empty(mods_u8.shape, dtype=torch.uint8, pin_memory=True)
        host.copy_(mods_u8, non_blocking=True)
        return {"mods": host}
