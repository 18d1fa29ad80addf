"""Batch multi-style stylisation: the reference's per-file loop (batch_process_images.py:498-531 --
one image per iteration, B=1) and its output-space style blends (advanced_transform.py:206-213,
direct_transform.py:155-165, batch_process_images.py:306-309) as ONE batched device pipeline.

"Multi-style with adjustable weights" in the reference is a linear blend of generator outputs
(SURVEY.md F4):  out = gain * (sum_s w_s * G_s(x) + w_x * x).  Each style s is one generator
(one state_dict).  Images are independent (InstanceNorm is per-sample, LocalAttention per-window),
so a batch is sharded by image across GPUs with no communication (shard_range below).

The batch is walked in micro-batches (default 16 images: measured best on B200 -- large enough to
amortise the persistent kernels' ramp-up/tail and the small-plane launches, small enough to bound the
activation footprint); host input is staged through pinned memory on a copy stream so H2D of
micro-batch i+1 overlaps the compute of micro-batch i.
"""
import math
import os

import torch

from . import _lib, ops


def check_blend_args(S, B, H, W, weights, w_x, weight_maps, feather_sigma):
    """Validates the blend arguments of MultiStyleStylizer.__call__ for S styles and B images of HxW before any device work:
    exactly one of `weights` (S global weights) and `weight_maps` (fp [Bm, K, h, w], Bm in {1, B}, K in {S, S+1}, h <= H,
    w <= W; map S weights the input image, so w_x must be 0) and a finite feather_sigma >= 0.  Raises ValueError."""
    if (weights is None) == (weight_maps is None):
        raise ValueError("give exactly one of `weights` (global) and `weight_maps` (per pixel)")
    if weight_maps is None:
        if len(weights) != S:
            raise ValueError(f"{S} styles but {len(weights)} weights")
        return
    if w_x != 0.0:
        raise ValueError("w_x must be 0 with weight_maps: map S (of S+1) weights the input image")
    if not torch.is_tensor(weight_maps) or not weight_maps.is_floating_point():
        raise ValueError("weight_maps must be a floating-point tensor [Bm, K, h, w]")
    if weight_maps.dim() != 4:
        raise ValueError(f"weight_maps must be [Bm, K, h, w], got shape {tuple(weight_maps.shape)}")
    Bm, K, h, w = weight_maps.shape
    if K not in (S, S + 1):
        raise ValueError(f"{K} weight maps for {S} styles: need {S} (styles) or {S + 1} (styles and the input image)")
    if Bm not in (1, B):
        raise ValueError(f"{Bm} map sets for {B} images: need 1 (shared) or {B} (one per image)")
    if not (1 <= h <= H and 1 <= w <= W):
        raise ValueError(f"{h}x{w} weight maps for {H}x{W} images: maps must be non-empty and no larger than the image")
    if not math.isfinite(feather_sigma) or feather_sigma < 0:
        raise ValueError(f"feather_sigma must be finite and >= 0, got {feather_sigma}")


def shard_range(num_images, rank, world_size):
    """Contiguous shard [lo, hi) of `num_images` images for `rank` (no communication needed)."""
    per = (num_images + world_size - 1) // world_size
    lo = min(rank * per, num_images)
    return lo, min(lo + per, num_images)


class MultiStyleStylizer:
    def __init__(self, generators, precision="bf16", micro_batch=32, style_streams=None, use_graph=None):
        if not generators:
            raise ValueError("need at least one generator (one per style)")
        self.generators = list(generators)
        for g in self.generators:
            g.eval()
            g.set_precision(precision)
        self.micro_batch = int(micro_batch)
        self.device = next(self.generators[0].parameters()).device
        self._copy_stream = None
        # The S forwards of a micro-batch are independent until the blend: each style runs on its own stream, so the
        # HBM-bound kernels of one style (1x1 convs, IN apply) overlap the shared-memory / issue-bound ones of another
        # (MultiScaleBlock branches, LocalAttention) and one style's kernel tails are filled by the next one's CTAs.
        if style_streams is None:
            style_streams = os.environ.get("MSG_STYLE_STREAMS", "1") == "1"
        self.style_streams = bool(style_streams) and len(self.generators) > 1
        self._streams = None
        if use_graph is None:
            use_graph = os.environ.get("MSG_STYLE_GRAPH", "1") == "1"
        self.use_graph = bool(use_graph)
        self._graphs = {}

    def _forward_chunk(self, xi, weights, w_x, gain, clip, dst, maps=None, normalize=False, style=None):
        """All styles of one micro-batch + the blend into dst, enqueued on the current stream (and the style streams).
        maps: the micro-batch's weight maps [Bm, K, h, w] on the device (per-pixel blend) instead of `weights`.
        style: the micro-batch's style mix ([S] or [Bi, S] on the device) for conditional generators."""
        cur = torch.cuda.current_stream(self.device)
        capturing = torch.cuda.is_current_stream_capturing()
        if self.style_streams:
            if self._streams is None:
                self._streams = [torch.cuda.Stream(self.device) for _ in self.generators]
            ready = torch.cuda.Event()
            ready.record(cur)                     # xi staged, previous micro-batch's blend enqueued
            ys, done = [], []
            for g, st in zip(self.generators, self._streams):
                st.wait_event(ready)
                with torch.cuda.stream(st):
                    y = g(xi) if style is None else g(xi, style=style)
                    ev_s = torch.cuda.Event()
                    ev_s.record(st)
                if not capturing:                 # (inside a capture the graph's private pool orders reuse itself)
                    xi.record_stream(st)
                    if style is not None:
                        style.record_stream(st)
                    y.record_stream(cur)
                ys.append(y)
                done.append(ev_s)
            for ev_s in done:
                cur.wait_event(ev_s)
        else:
            ys = [g(xi) if style is None else g(xi, style=style) for g in self.generators]
        if maps is None:
            ops.blend_outputs(ys, weights, x=xi if w_x != 0.0 else None, w_x=w_x, gain=gain, clip=clip, out=dst)
        else:
            ops.blend_maps(ys, maps, x=xi if maps.shape[1] > len(ys) else None, gain=gain, clip=clip, normalize=normalize,
                           out=dst)

    def _replay(self, xi, weights, w_x, gain, clip, dst, pver=None, maps=None, normalize=False, style=None):
        """CUDA-graph path: the ~210 launches of a micro-batch (S forwards + blend) are captured once per
        (shape, blend parameters) and replayed, so the host cost of a micro-batch is one graph launch.  Weights are
        read through the per-generator pack caches at capture time: `invalidate_graphs()` after changing them.
        Weight maps are a graph input like the images: the key holds their shape and `normalize`, each replay copies the
        micro-batch's maps into the entry's static buffer.  So is the style mix of conditional generators: moving a style
        slider replays the same graph."""
        key = (tuple(xi.shape), tuple(float(w) for w in weights) if maps is None else ("maps", tuple(maps.shape), bool(normalize)),
               float(w_x), float(gain), clip, dst.dtype,
               pver if pver is not None else tuple(g.param_version() for g in self.generators),
               None if style is None else ("style", tuple(style.shape)))
        ent = self._graphs.get(key)
        if ent is None:
            sx = torch.empty_like(xi)
            sd = torch.empty_like(dst)
            sx.copy_(xi)
            sm = None if maps is None else maps.clone()
            ss = None if style is None else style.clone()
            for _ in range(2):                    # warm-up outside capture: weight packs, function attributes, allocator
                self._forward_chunk(sx, weights, w_x, gain, clip, sd, sm, normalize, ss)
            torch.cuda.current_stream(self.device).synchronize()
            gr = torch.cuda.CUDAGraph()
            l0 = _lib.launches
            try:
                with torch.cuda.graph(gr):
                    self._forward_chunk(sx, weights, w_x, gain, clip, sd, sm, normalize, ss)
            except Exception as e:                # capture refused (e.g. a user-supplied transformer block that syncs):
                import warnings                   # same kernels, launched one by one
                warnings.warn(f"MultiStyleStylizer: CUDA-graph capture failed ({e!r}); continuing without graphs")
                self.use_graph = False
                torch.cuda.synchronize(self.device)
                self._forward_chunk(xi, weights, w_x, gain, clip, dst, maps, normalize, style)
                return
            while len(self._graphs) >= 8:         # stale keys (old parameter versions, other shapes): drop the oldest
                self._graphs.pop(next(iter(self._graphs)))
            # the captured launches address the packed weights of each generator's cache (allocated during the warm-up, outside
            # the graph's pool): the entry keeps them alive, so invalidate_packed_weights() cannot free memory a graph reads
            keep = [list(g._engine._cache.values()) for g in self.generators]
            ent = self._graphs[key] = (gr, sx, sd, _lib.launches - l0, keep, sm, ss)
        gr, sx, sd, n_launches, _, sm, ss = ent
        sx.copy_(xi)
        if sm is not None:
            sm.copy_(maps)
        if ss is not None:
            ss.copy_(style)
        gr.replay()
        _lib.launches += n_launches               # kernels inside the replayed graph (the launch counter is per C-ABI call)
        dst.copy_(sd)

    def invalidate_graphs(self):
        self._graphs.clear()

    @torch.no_grad()
    def __call__(self, x, weights=None, w_x=0.0, gain=1.0, clip=None, out_uint8=False, out=None, *, weight_maps=None,
                 feather_sigma=0.0, normalize_maps=False, style=None):
        """x: float32 [B,3,H,W] in [-1,1], or uint8 [B,H,W,3] (PIL layout: ToTensor + Normalize(0.5, 0.5) then run on the
        device, batch_process_images.py:287-291 -- a quarter of the host-to-device bytes), on the device or on the host
        (pinned for overlap).
        Returns the blended fp32 images [B,3,H,W] on the device, or -- with out_uint8=True -- the
        uint8 images ((v+1)/2 -> clamp -> *255, direct_transform.py:66-71) in `out` (host or device
        uint8 tensor [B,3,H,W]; allocated on the device if None).
        weight_maps (instead of `weights`): per-pixel style weights [Bm, K, h, w] (host or device, Bm in {1, B}, K in {S, S+1}
        with map S weighting the input image, h <= H, w <= W), sampled bilinearly at every pixel (ops.blend_maps;
        enhanced_local_style.py:126-176, 232-236).  A [B, S, 1, 1] tensor gives each image its own global mix.
        feather_sigma > 0 blurs each map plane with a Gaussian first (ops.gaussian_blur); normalize_maps divides the
        sampled weights of each pixel by their sum.
        style (style-conditional generators, EnhancedGenerator.enable_style_affine, all with the same number of styles K):
        the mix fp32 [K] or [B, K] every generator runs with (sliced per micro-batch like the weight maps)."""
        S = len(self.generators)
        hw = (tuple(x.shape[1:3]) if x.dtype == torch.uint8 else tuple(x.shape[2:4])) if x.dim() == 4 else (0, 0)
        check_blend_args(S, x.shape[0], *hw, weights, w_x, weight_maps, float(feather_sigma))
        num_styles = {getattr(g, "num_styles", None) for g in self.generators}
        if len(num_styles) != 1:
            raise ValueError("the generators must all be plain, or all style-conditional with the same number of styles")
        if style is not None or num_styles != {None}:
            style = self.generators[0]._style_mix(style, x)
        with torch.cuda.device(self.device):
            if style is not None:
                style = style.to(self.device).contiguous()
            maps = None
            if weight_maps is not None:            # moved and feathered once per call, sliced per micro-batch
                maps = weight_maps.to(self.device, torch.float32).contiguous()
                if feather_sigma > 0:
                    maps = ops.gaussian_blur(maps, feather_sigma)
            return self._run(x, weights, w_x, gain, clip, out_uint8, out, maps, bool(normalize_maps), style)

    def _run(self, x, weights, w_x, gain, clip, out_uint8, out, maps=None, normalize=False, style=None):
        B = x.shape[0]
        mb = self.micro_batch
        host_in = not x.is_cuda
        u8_in = x.dtype == torch.uint8
        if u8_in and (x.dim() != 4 or x.shape[3] != 3):
            raise RuntimeError("MultiStyleStylizer: uint8 input must be [B,H,W,3]")
        hw = tuple(x.shape[1:3]) if u8_in else tuple(x.shape[2:])
        if out is None:
            out = torch.empty((B, 3) + hw, device=self.device,
                              dtype=torch.uint8 if out_uint8 else torch.float32)
        host_out = not out.is_cuda
        cur = torch.cuda.current_stream(self.device)
        if host_in and self._copy_stream is None:
            self._copy_stream = torch.cuda.Stream(self.device)
        chunks = [(lo, min(lo + mb, B)) for lo in range(0, B, mb)]
        pver = tuple(g.param_version() for g in self.generators) if self.use_graph else None   # once per call, not per chunk
        staged = {}

        def stage(i):
            lo, hi = chunks[i]
            if not host_in:
                staged[i] = (x[lo:hi], None)
                return
            with torch.cuda.stream(self._copy_stream):
                t = x[lo:hi].to(self.device, non_blocking=True)
                ev = torch.cuda.Event()
                ev.record(self._copy_stream)
            staged[i] = (t, ev)

        stage(0)
        for i, (lo, hi) in enumerate(chunks):
            if i + 1 < len(chunks):
                stage(i + 1)
            xi, ev = staged.pop(i)
            if ev is not None:
                cur.wait_event(ev)
                xi.record_stream(cur)
            if u8_in:
                xi = ops.u8_canvas_to_nchw(xi.contiguous())
            dst = None if host_out else out[lo:hi]      # device result: the blend writes it in place
            if dst is None:
                dst = torch.empty((hi - lo,) + tuple(out.shape[1:]), device=self.device, dtype=out.dtype)
            mi = None if maps is None else (maps if maps.shape[0] == 1 else maps[lo:hi])
            si = None if style is None else (style if style.dim() == 1 else style[lo:hi])
            if self.use_graph:
                self._replay(xi, weights, w_x, gain, clip, dst, pver, mi, normalize, si)
            else:
                self._forward_chunk(xi, weights, w_x, gain, clip, dst, mi, normalize, si)
            if host_out:
                out[lo:hi].copy_(dst, non_blocking=True)
        if host_out:
            # the D2H copies into a (pinned) host tensor are asynchronous: the caller is about to read / save the images,
            # so the call returns only when the last copy has landed (one event wait, not a device-wide synchronize)
            done = torch.cuda.Event()
            done.record(cur)
            done.synchronize()
        return out
