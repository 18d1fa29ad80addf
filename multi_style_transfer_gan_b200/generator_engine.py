"""Forward / backward schedule of the EnhancedGenerator on the msg_b200 kernels.

Follows enhanced_generator.py:86-228 of the reference (module structure :91-147, forward
:211-228).  The engine works on a flat ``{state_dict key: fp32 tensor}`` view of the parameters and
NHWC activations; it owns no parameters itself.

Per stage (down1/down2/up1/up2, width C), kernels launched in the forward:
    main conv (4x4 s2 conv | 4 phases of the 4x4 s2 convT)  + IN statistics in the epilogue
    IN apply + ReLU
    qkv 1x1 conv -> LocalAttention core -> proj 1x1 conv
    4 branch convs writing channel slices of ONE [N,H,W,C] tensor (no cat) + shared IN statistics
    IN apply + ReLU -> fusion 1x1 conv (+ statistics) -> IN apply + ReLU + residual add
"""
import os

import torch
import torch.nn.functional as F

from . import ops, slab
from .ops import ACT_NONE, ACT_RELU, ACT_TANH, ConvGeom

STAGES = ("down1", "down2", "up1", "up2")
BRANCHES = ((1, 0, 1), (3, 1, 1), (3, 2, 2), (3, 4, 4))  # (k, pad, dil) of branch1..4, :52-71


def _pad_dim(t, dim, to):
    if t.shape[dim] == to:
        return t
    pad = [0, 0] * (t.dim() - dim - 1) + [0, to - t.shape[dim]]
    return F.pad(t, pad)


class _StatsArena:
    """All InstanceNorm statistics buffers ([N, C, 2] fp64 raw sums) of one encode / decode call come from ONE zeroed
    allocation: one fill launch instead of one per normalised tensor (13 per forward)."""

    def __init__(self, N, channels_total, device):
        self.buf = torch.zeros(N * channels_total * 2, device=device, dtype=torch.float64)
        self.N, self.pos = N, 0

    def take(self, C):
        n = self.N * C * 2
        if self.pos + n > self.buf.numel():          # (not expected: sized from the stage widths)
            return torch.zeros((self.N, C, 2), device=self.buf.device, dtype=torch.float64)
        t = self.buf[self.pos:self.pos + n].view(self.N, C, 2)
        self.pos += n
        return t


def norm_sites(c):
    """The 13 InstanceNorm apply sites of a generator of width c in forward order: (site, channels, affine holders).  The four
    branch norms of a MultiScaleBlock are one apply over the concatenated branches, so their holders share one site, in branch
    order."""
    width = {"down1": 2 * c, "down2": 4 * c, "up1": 2 * c, "up2": c}
    sites = [("initial.1", c, ("initial.1",))]
    for s in STAGES:
        C = width[s]
        sites += [(f"{s}.1", C, (f"{s}.1",)),
                  (f"{s}.4.branch", C, tuple(f"{s}.4.branch{i}.1" for i in range(1, 5))),
                  (f"{s}.4.fusion.1", C, (f"{s}.4.fusion.1",))]
    return sites


class StyleAffine:
    """Per-image InstanceNorm affines of one conditional forward: the mix w [N, S] and the tables gamma / beta [N, Ct] fp32 that
    msg_style_affine built from it, one column range per norm site (`off`).  The backward of the same forward reads them again
    (checkpointed recompute included) and collects the per-image affine gradients of all sites in one fp64 arena `sums`."""

    def __init__(self, w, gamma, beta, off):
        self.w, self.gamma, self.beta, self.off = w, gamma, beta, off
        self.sums = None

    def at(self, site):
        """(gamma, beta, img_stride) of a site, the C-ABI's affine argument (include/msg_b200.h)"""
        o = self.off[site]
        return self.gamma.view(-1)[o:], self.beta.view(-1)[o:], self.gamma.shape[1]

    def sums_at(self, site):
        return self.sums[2 * self.off[site]:]


def _site(A, name):
    return None if A is None else A.at(name)


class GradSink(dict):
    """Parameter gradients accumulated straight into caller-owned fp32 buffers -- the views of the optimizer's flat gradient
    buffer -- instead of fresh tensors that autograd then adds to .grad: per conv that was a zeros() for the packed gradient, a
    zeros() for the unpacked one, the unpack, a dict add and autograd's accumulate (~1900 small launches per train step).  The
    packed gradients of one backward come from ONE zeroed arena."""

    def __init__(self, sinks, arena_floats, device):
        super().__init__()
        self.sinks = sinks
        self.arena = torch.zeros(arena_floats, device=device, dtype=torch.float32) if arena_floats else None
        self.pos, self.used = 0, 0

    def scratch(self, n, device):
        n = (n + 63) // 64 * 64             # (keeps every slice 256-byte aligned: the wgrad kernel reduces in 16-byte rows)
        self.used += n
        if self.arena is None or self.pos + n > self.arena.numel():
            return torch.zeros(n, device=device, dtype=torch.float32)
        t = self.arena[self.pos:self.pos + n]
        self.pos += n
        return t


class GeneratorEngine:
    def __init__(self, channels):
        c = self.c = channels
        if c % 4:
            raise ValueError("EnhancedGenerator: channels must be a multiple of 4 (MultiScaleBlock splits C/4)")
        # image channels 3 -> 4 (fp32) / 8 (bf16: the tcgen05 gather moves 16-byte chunks), with zero
        # weights for the pad channels; output conv 3 -> 4 / 8 filters (extra ones zero, never stored)
        self.width = {"down1": 2 * c, "down2": 4 * c, "up1": 2 * c, "up2": c}
        self.inwidth = {"down1": c, "down2": 2 * c, "up1": 4 * c, "up2": 2 * c}
        g = self.geom = {}
        for pad in (4, 8):
            g[f"initial.0@{pad}"] = ConvGeom("conv", pad, c, 7, 1, 3)
            g[f"output.0@{pad}"] = ConvGeom("conv", c, pad, 7, 1, 3)
        for s in STAGES:
            C, Ci = self.width[s], self.inwidth[s]
            g[f"{s}.0"] = ConvGeom("convT" if s.startswith("up") else "conv", Ci, C, 4, 2, 1)
            g[f"{s}.3.qkv"] = ConvGeom("conv", C, 3 * C, 1)
            g[f"{s}.3.proj"] = ConvGeom("conv", C, C, 1)
            for i, (k, p, d) in enumerate(BRANCHES, start=1):
                g[f"{s}.4.branch{i}.0"] = ConvGeom("conv", C, C // 4, k, 1, p, d)
            g[f"{s}.4.fusion.0"] = ConvGeom("conv", C, C, 1)
        self._cache = {}
        # row-slab programs (bf16 path, widths that are multiples of 64): fused MSB branches, 7x7 convs
        self.use_slab = True
        def fits(build):
            # a program that exceeds the descriptor's tap / K-block tables (wide generators: C = 512 at c = 128) is simply not
            # offered: those layers take the per-tap TMA kernel
            try:
                return build()
            except ValueError:
                return None
        widths = sorted(C for C in set(self.width.values()) if C % 64 == 0)
        self._msb_prog = {C: pr for C in widths for pr in [fits(lambda: slab.msb_program(C))] if pr is not None}
        self._msb_dprog = {C: pr for C in widths for pr in [fits(lambda: slab.msb_dgrad_program(C))] if pr is not None}
        self._in_prog = fits(lambda: slab.conv7_in_program(c)) if c % 16 == 0 else None
        self._out_prog = fits(lambda: slab.conv7_out_shift_program(c)) if c % 64 == 0 else None     # taps-as-N (conv_shift.cu)
        self._msb64_prog = slab.msb64_shift_program()
        self._convT_prog = {s: pr for s in ("up1", "up2") if self.inwidth[s] % 64 == 0 and self.width[s] % 16 == 0
                            for pr in [fits(lambda: slab.convT_phase_programs(self.inwidth[s], self.width[s]))] if pr is not None}
        self.convT_slab = os.environ.get("MSG_CONVT_SLAB", "1") == "1"
        self.msb64_taps_as_n = os.environ.get("MSG_MSB64_SHIFT", "0") == "1"
        # Row-ring kernel for the C = 64 branches (csrc/msb_ring.cu): 0.48 ms per 16 images at 512^2 vs 0.67 ms for the per-tap slab
        # kernel (profiles/r2_msb_ring.md).  MSG_MSB64_RING=0 falls back to the latter.
        self.msb64_ring = os.environ.get("MSG_MSB64_RING", "1") == "1"
        # ... and for the C = 128 branches (three passes): 0.27 ms vs 0.38 ms per 16 images at 256^2.  MSG_MSB128_RING=0 falls back.
        self.msb128_ring = os.environ.get("MSG_MSB128_RING", "1") == "1"
        # ... and for the 128 -> 64 transposed conv of up2 (csrc/convt_ring.cu).  MSG_CONVT_RING=0 falls back to the phase slabs.
        self.convT_ring = os.environ.get("MSG_CONVT_RING", "1") == "1"
        # ... and for the output conv fused with the IN + ReLU + residual in front of it (csrc/out7_ring.cu).  MSG_OUT7_RING=0 falls back.
        self.out7_ring = os.environ.get("MSG_OUT7_RING", "1") == "1"
        # ... and for down1's 4x4 stride-2 conv fused with the input layer's IN + ReLU (csrc/down_ring.cu).  MSG_DOWN_RING=0 falls back.
        self.down_ring = os.environ.get("MSG_DOWN_RING", "1") == "1"
        self.fuse_in_norm = os.environ.get("MSG_FUSE_IN_NORM", "1") == "1"
        self.fuse_la = os.environ.get("MSG_FUSE_LA", "1") == "1"      # fused LocalAttention stage kernel (inference)
        self._arena_floats = 0          # packed-gradient floats of one backward (measured on the first one)
        # style-conditional models (EnhancedGenerator.enable_style_affine): column ranges of the norm sites in the affine tables
        self.sites = norm_sites(c)
        self.site_off, self.Ct = {}, 0
        for name, C, _ in self.sites:
            self.site_off[name] = self.Ct
            self.Ct += C

    def _versions(self, params, names):
        return tuple((params[n].data_ptr(), params[n]._version) for n in names)

    def _slab_cached(self, params, key, names, build):
        ver = self._versions(params, names)
        hit = self._cache.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        t = build()
        self._cache[key] = (ver, t)
        return t

    @staticmethod
    def edge_pad(dtype):
        return 4 if dtype == torch.float32 else 8

    def _g(self, name, dtype):
        if name in ("initial.0", "output.0"):
            return self.geom[f"{name}@{self.edge_pad(dtype)}"]
        return self.geom[name]

    # ---- packed-weight cache ---------------------------------------------------------------------
    def invalidate(self):
        self._cache.clear()

    def _master(self, params, name, dtype):
        w = params[f"{name}.weight"]
        if name == "initial.0":
            w = _pad_dim(w, 1, self.edge_pad(dtype))
        elif name == "output.0":
            w = _pad_dim(w, 0, self.edge_pad(dtype))
        return w.contiguous()

    def _packed(self, params, name, which, dtype):
        w = params[f"{name}.weight"]
        key = (name, which, dtype)
        ver = (w.data_ptr(), w._version)
        hit = self._cache.get(key)
        if hit is not None and hit[0] == ver:
            return hit[1]
        m = self._master(params, name, dtype)
        g = self._g(name, dtype)
        t = g.pack_fwd(m, dtype) if which == "fwd" else g.pack_dgrad(m, dtype)
        self._cache[key] = (ver, t)
        return t

    def _bias(self, params, name, dtype=None):
        b = params[f"{name}.bias"]
        if name == "output.0":
            b = _pad_dim(b, 0, self.edge_pad(dtype))
        return b.contiguous()

    # ---- style affine --------------------------------------------------------------------------
    def _holder_columns(self):
        """(holder, first column, channels) of the 25 affine holders in table order"""
        for name, C, holders in self.sites:
            q = C // len(holders)
            for i, h in enumerate(holders):
                yield h, self.site_off[name] + i * q, q

    def style_tables(self, P, w):
        """w: fp32 [N, S] mix on the device -> StyleAffine (one msg_style_affine launch).  The holders' [S, C] parameters are
        packed into [S, Ct] once per parameter version, like the weight packs."""
        hs = [h for h, _, _ in self._holder_columns()]
        tabs = []
        for which in ("weight", "bias"):
            names = [f"{h}.{which}" for h in hs]
            tabs.append(self._slab_cached(P, ("style_affine", which), names,
                                          lambda: torch.cat([P[k].detach() for k in names], 1).contiguous()))
        g, b = ops.style_affine(w, *tabs)
        return StyleAffine(w, g, b, self.site_off)

    def style_affine_begin_bwd(self, A):
        A.sums = torch.zeros(A.w.shape[0] * self.Ct * 2, device=A.w.device, dtype=torch.float64)

    def style_affine_end_bwd(self, G, A):
        """One msg_style_affine_bwd over the backward's sums arena -> the [S, C] gradients of the holders into G."""
        S = A.w.shape[1]
        dg = torch.zeros((S, self.Ct), device=A.w.device, dtype=torch.float32)
        db = torch.zeros_like(dg)
        ops.style_affine_bwd(A.sums, A.w, dg, db)
        A.sums = None
        for h, o, q in self._holder_columns():
            for k, t in ((f"{h}.weight", dg[:, o:o + q]), (f"{h}.bias", db[:, o:o + q])):
                if isinstance(G, GradSink):
                    G.sinks[k].add_(t)
                else:
                    G[k] = t if k not in G else G[k] + t

    def _in_bwd(self, x, st, dy, A, site):
        """Backward of ReLU(IN(x)) at one norm site; conditional: reduce -> apply with the forward's per-image affine, the
        reductions (d beta_n, d gamma_n) landing in the site's columns of the sums arena."""
        if A is None:
            return ops.instnorm_bwd(x, st, dy, ACT_RELU)
        aff, sums = A.at(site), A.sums_at(site)
        ops.instnorm_bwd_reduce_affine(x, st, dy, aff, sums, ACT_RELU)
        return ops.instnorm_bwd_apply_affine(x, st, dy, sums, aff, ACT_RELU)

    # ---- forward ---------------------------------------------------------------------------------
    def _stage_fwd(self, P, s, a_in, dtype, keep=True, arena=None, defer_apply=False, A=None):
        """keep=False (inference): intermediates are dropped as soon as their consumer has been
        launched, so the caching allocator recycles them within the stage."""
        g = self.geom
        C = self.width[s]
        x_in = a_in[0] if isinstance(a_in, tuple) else a_in       # (a tuple: raw conv output + its statistics, normalised by the consumer)
        N = x_in.shape[0]
        dev = x_in.device
        if arena is None:
            arena = _StatsArena(N, 3 * C, dev)
        st0 = arena.take(C)
        if isinstance(a_in, tuple):
            # inference, c = 64: the IN + ReLU of the 7x7 input layer is applied by this stage's 4x4 stride-2 conv on its landed row
            # slabs (csrc/down_ring.cu: 0.50 -> ~0.3 ms per 16 images for apply + conv, the normalised tensor never exists in HBM)
            yi, sti = a_in
            wn = f"{s}.0.weight"
            wsl = self._slab_cached(P, (s, "down_ring_w"), [wn], lambda: slab.down_ring_weights(P[wn].detach()))
            y0 = slab.down_ring(yi, sti, wsl, self._bias(P, f"{s}.0"), C, stats=st0, in_affine=_site(A, "initial.1"))
        elif (self.convT_ring and g[f"{s}.0"].kind == "convT" and dtype == torch.bfloat16 and self.inwidth[s] in (64, 128) and C % 64 == 0):
            # transposed conv as a row ring of TMEM accumulators (csrc/convt_ring.cu): one launch per horizontal output phase, every
            # input row loaded once per launch, the four vertical taps of a horizontal tap as one N = 256 MMA.  128 -> 64 at 256^2:
            # 0.27 ms per 16 images vs 0.46 ms for the four row-slab phase launches (1.0 PFLOP/s, 0.71 of the sustained bf16 peak)
            wn = f"{s}.0.weight"
            wsl = self._slab_cached(P, (s, "convT_ring_w"), [wn], lambda: slab.convt_ring_weights(P[wn].detach()))
            y0 = torch.empty((N, 2 * a_in.shape[1], 2 * a_in.shape[2], C), device=dev, dtype=dtype)
            slab.convt_ring(a_in, wsl, self._bias(P, f"{s}.0"), C, out=y0, stats=st0)
        elif (self.convT_slab and s in self._convT_prog and g[f"{s}.0"].kind == "convT" and dtype == torch.bfloat16 and self.inwidth[s] % 64 == 0 and
                C % 16 == 0 and C * self.inwidth[s] <= 64 * 128 and a_in.shape[2] % 8 == 0):
            # (weights of a phase resident in shared memory: 128 -> 64 measured 0.64 -> 0.49 ms per 16 images at 256^2;
            #  with streamed weights, 256 -> 128, the per-tap TMA kernel is as fast: 0.36 vs 0.38 ms)
            # transposed conv as four row-slab programs (each input row slab read once per phase for both horizontal taps)
            progs = self._convT_prog[s]
            wsl = self._slab_cached(P, (s, "convT_w"), [f"{s}.0.weight"],
                                    lambda: slab.convT_phase_weight_slabs(progs, self._packed(P, f"{s}.0", "fwd", dtype), self.inwidth[s], C))
            y0 = torch.empty((N, 2 * a_in.shape[1], 2 * a_in.shape[2], C), device=dev, dtype=dtype)
            slab.convT_slab(progs, a_in, wsl, self._bias(P, f"{s}.0"), y0, stats=st0)
        else:
            y0 = g[f"{s}.0"].forward(a_in, self._packed(P, f"{s}.0", "fwd", dtype), self._bias(P, f"{s}.0"), stats=st0)
        wq = self._packed(P, f"{s}.3.qkv", "fwd", dtype)
        wp = self._packed(P, f"{s}.3.proj", "fwd", dtype)
        if not keep and self.fuse_la and ops.la_stage_supported(y0, wq, wp):
            # inference, C in {64, 128}: the whole LocalAttention stage -- IN + ReLU of y0 on the landed tile, qkv 1x1, window
            # attention with S / P in tensor memory, proj 1x1 -- is ONE tcgen05 launch; qkv and the attention output never
            # exist in HBM (csrc/la_stage.cu)
            a1 = ops.la_stage_fwd(y0, wq, self._bias(P, f"{s}.3.qkv"), wp, self._bias(P, f"{s}.3.proj"), in_stats=st0, in_act=ACT_RELU,
                                  in_affine=_site(A, f"{s}.1"))
            del y0
            return self._msb_fwd(P, s, a1, None, dtype, keep, arena, g, C, defer_apply, A)
        if not keep and self.fuse_in_norm and g[f"{s}.3.qkv"].fused_in_norm_ok(y0, wq):
            # inference: ReLU(IN(y0)) has ONE consumer, the 1x1 qkv conv (LocalAttention has no residual), so the
            # conv normalises its A tiles in shared memory and the normalised tensor never exists in HBM
            a0 = None
            qkv = g[f"{s}.3.qkv"].forward(y0, wq, self._bias(P, f"{s}.3.qkv"), in_stats=st0, in_act=ACT_RELU,
                                          in_affine=_site(A, f"{s}.1"))
        else:
            a0 = ops.instnorm_apply(y0, st0, ACT_RELU, out=None if keep else y0, affine=_site(A, f"{s}.1"))
            qkv = g[f"{s}.3.qkv"].forward(a0, wq, self._bias(P, f"{s}.3.qkv"))
        att = ops.local_attn_fwd(qkv)
        if not keep:
            del y0, a0, qkv
        a1 = g[f"{s}.3.proj"].forward(att, wp, self._bias(P, f"{s}.3.proj"))
        if not keep:
            del att
            return self._msb_fwd(P, s, a1, None, dtype, keep, arena, g, C, defer_apply, A)
        return self._msb_fwd(P, s, a1, dict(a_in=a_in, y0=y0, st0=st0, a0=a0, qkv=qkv, att=att), dtype, keep, arena, g, C, A=A)

    def _msb_fwd(self, P, s, a1, saved, dtype, keep, arena, g, C, defer_apply=False, A=None):
        """MultiScaleBlock of stage s on a1 (enhanced_generator.py:78-84)."""
        dev = a1.device
        b = torch.empty_like(a1)
        stb = arena.take(C)
        if self.use_slab and dtype == torch.bfloat16 and C in self._msb_prog and a1.shape[2] % 8 == 0:
            # one launch for the 1x1 + 3x3 dil 1/2/4 branches: they share each input-row slab
            wn = [f"{s}.4.branch{i}.0.weight" for i in range(1, 5)]
            bn_ = [f"{s}.4.branch{i}.0.bias" for i in range(1, 5)]
            bsl = self._slab_cached(P, (s, "msb_b"), bn_, lambda: torch.cat([P[k].detach() for k in bn_]).contiguous())
            if (C == 64 and self.msb64_ring) or (C == 128 and self.msb128_ring):
                # row ring of TMEM accumulators (csrc/msb_ring.cu): every input row loaded once, vertical taps stacked along N
                # (one launch at C = 64, three passes at C = 128)
                wsl = self._slab_cached(P, (s, "msb_ring_w"), wn, lambda: slab.msb_ring_weights([P[k].detach() for k in wn], C))
                slab.msb_ring(a1, wsl, bsl, C, out=b, stats=stb)
            elif C == 64 and self.msb64_taps_as_n:   # taps-as-N (conv_shift.cu): 1.09 ms vs 0.89 ms per 16 images at
                # 512^2 for the per-tap slab kernel once its issue loop went lean, so off by default
                wsl = self._slab_cached(P, (s, "msb_w"), wn, lambda: slab.msb64_shift_weights([P[k].detach() for k in wn]))
                slab.conv_shift(self._msb64_prog, a1, wsl, bsl, out=b, stats=stb)
            else:           # one MMA per tap on shifted views of the slab (conv_slab.cu)
                prog = self._msb_prog[C]
                wsl = self._slab_cached(P, (s, "msb_w"), wn, lambda: slab.msb_weight_slab(prog, [P[k].detach() for k in wn]))
                slab.conv_slab(prog, a1, wsl, bsl, out=b, stats=stb)
        else:
            for i in range(1, 5):
                n = f"{s}.4.branch{i}.0"
                g[n].forward(a1, self._packed(P, n, "fwd", dtype), self._bias(P, n), out=b, co_off=(i - 1) * (C // 4), stats=stb)
        stf = arena.take(C)
        n = f"{s}.4.fusion.0"
        wf = self._packed(P, n, "fwd", dtype)
        if not keep and self.fuse_in_norm and g[n].fused_in_norm_ok(b, wf):
            bn = None       # ReLU(IN(branches)) is consumed only by the 1x1 fusion conv: normalised on the fly
            f = g[n].forward(b, wf, self._bias(P, n), stats=stf, in_stats=stb, in_act=ACT_RELU, in_affine=_site(A, f"{s}.4.branch"))
        else:
            bn = ops.instnorm_apply(b, stb, ACT_RELU, out=None if keep else b, affine=_site(A, f"{s}.4.branch"))
            f = g[n].forward(bn, wf, self._bias(P, n), stats=stf)
        if defer_apply and not keep:
            # the stage's last IN + ReLU + residual is applied by its consumer on the landed row slabs (csrc/out7_ring.cu)
            return (f, stf, a1), None
        a2 = ops.instnorm_apply(f, stf, ACT_RELU, residual=a1, out=None if keep else f, affine=_site(A, f"{s}.4.fusion.1"))
        if not keep:
            return a2, None
        saved.update(a1=a1, b=b, stb=stb, bn=bn, f=f, stf=stf)
        return a2, saved

    def encode(self, P, x, dtype, save, A=None):
        """x: fp32 NCHW image -> (a [N,H/4,W/4,4c] NHWC, saved).  A: the StyleAffine of a conditional model, else None."""
        N, Cx, H, W = x.shape
        if Cx != 3:
            raise RuntimeError(f"EnhancedGenerator expects 3 input channels, got {Cx}")
        if H % 16 or W % 16:
            # the reference's LocalAttention pad path is broken (enhanced_generator.py:15-23): such
            # sizes raise there too (SURVEY.md 3.2).
            raise RuntimeError(f"EnhancedGenerator: H and W must be multiples of 16, got {H}x{W}")
        x0 = ops.nchw_to_nhwc(x, dtype, self.edge_pad(dtype))
        arena = _StatsArena(N, self.c + 3 * (self.width["down1"] + self.width["down2"]), x.device)
        sti = arena.take(self.c)
        if self.use_slab and dtype == torch.bfloat16 and self._in_prog is not None and W % 8 == 0:
            prog = self._in_prog
            wsl = self._slab_cached(P, ("initial", "slab_w"), ["initial.0.weight"],
                                    lambda: slab.conv7_in_weight_slab(prog, P["initial.0.weight"].detach()))
            yi = slab.conv_slab(prog, x0, wsl, self._bias(P, "initial.0"), stats=sti)
        else:
            yi = self._g("initial.0", dtype).forward(x0, self._packed(P, "initial.0", "fwd", dtype), self._bias(P, "initial.0"), stats=sti)
        if not save and self.down_ring and dtype == torch.bfloat16 and self.c == 64 and self.use_slab and H % 2 == 0 and W % 2 == 0:
            a = (yi, sti)           # applied by down1's first conv (csrc/down_ring.cu)
        else:
            a = ops.instnorm_apply(yi, sti, ACT_RELU, out=None if save else yi, affine=_site(A, "initial.1"))
        saved = {"x0": x0, "yi": yi, "sti": sti} if save else None
        for s in ("down1", "down2"):
            a_in = a
            a, sv = self._stage_fwd(P, s, a_in, dtype, keep=(save == "full"), arena=arena, A=A)
            if save:
                saved[s] = sv if save == "full" else {"a_in": a_in}
        return a, saved

    def decode(self, P, a, dtype, save, A=None):
        """a: [N,H/4,W/4,4c] NHWC -> (y fp32 NCHW in [-1,1], saved)."""
        saved = {} if save else None
        arena = _StatsArena(a.shape[0], 3 * (self.width["up1"] + self.width["up2"]), a.device)
        # inference at c = 64 (bf16): the output conv applies up2's last IN + ReLU + residual itself (one ring kernel instead of the
        # HBM-bound apply + the taps-as-N conv: csrc/out7_ring.cu)
        fuse_out = (not save and self.out7_ring and dtype == torch.bfloat16 and self.c == 64 and self.use_slab)
        for s in ("up1", "up2"):
            a_in = a
            a, sv = self._stage_fwd(P, s, a_in, dtype, keep=(save == "full"), arena=arena, defer_apply=(fuse_out and s == "up2"), A=A)
            if save:
                saved[s] = sv if save == "full" else {"a_in": a_in}
        if isinstance(a, tuple):
            f, stf, a1 = a
            N, H, W, _ = f.shape
            y = torch.empty((N, 3, H, W), device=f.device, dtype=torch.float32)
            wsl = self._slab_cached(P, ("output", "ring_w"), ["output.0.weight"], lambda: slab.out7_ring_weights(P["output.0.weight"].detach()))
            slab.out7_ring(f, stf, a1, wsl, P["output.0.bias"].detach().contiguous(), nchw_out=y, in_affine=_site(A, "up2.4.fusion.1"))
            return y, saved
        N, H, W, _ = a.shape
        y = torch.empty((N, 3, H, W), device=a.device, dtype=torch.float32)
        if self.use_slab and dtype == torch.bfloat16 and self._out_prog is not None and W % 8 == 0:
            prog = self._out_prog
            wsl = self._slab_cached(P, ("output", "slab_w"), ["output.0.weight"],
                                    lambda: slab.conv7_out_shift_weights(prog, P["output.0.weight"].detach()))
            slab.conv_shift(prog, a, wsl, P["output.0.bias"].detach().contiguous(), act=ACT_TANH, nchw_out=y)
        else:
            go = ConvGeom("conv", self.c, 3, 7, 1, 3)   # store 3 filters of the padded packed weight
            go.forward(a, self._packed(P, "output.0", "fwd", dtype), self._bias(P, "output.0", dtype), act=ACT_TANH, nchw_out=y)
        if save:
            saved["a_last"] = a
            saved["y"] = y
        return y, saved

    # ---- backward --------------------------------------------------------------------------------
    def _conv_bwd(self, P, G, name, x, dy, dtype, need_dx=True, in_hw=None, dy_c_off=0, dx_out=None, accumulate=False):
        """Accumulates weight / bias grads of conv `name` into G and returns dx (or None)."""
        g = self._g(name, dtype)
        m = self._master(P, name, dtype)
        sink = G.sinks if isinstance(G, GradSink) else None
        nb = m.shape[1] if g.kind == "convT" else m.shape[0]
        # A conv bias in front of an InstanceNorm has an EXACTLY zero gradient (the norm subtracts the plane mean: d(IN(y + b))/db
        # = 0; the reference's autograd produces ~1e-8 of rounding noise there).  Only the qkv / proj convs and the output conv
        # have live biases: the other 29 bias reductions of a generator backward are skipped (3.6 ms per train step).
        live_bias = name.endswith(".3.qkv") or name.endswith(".3.proj") or name == "output.0"
        padded = name in ("initial.0", "output.0")          # (weights zero-padded to 4 / 8 image channels: unpack via a temporary)
        direct = sink is not None and not padded
        dw = sink[f"{name}.weight"] if direct else torch.zeros_like(m)
        if not live_bias:
            db = None
        elif direct:
            db = sink[f"{name}.bias"]
        else:
            db = torch.zeros(nb, device=m.device, dtype=torch.float32)
        if name == "initial.0" and dtype == torch.bfloat16 and x.shape[3] == 8 and x.shape[2] % 8 == 0:
            # Cin = 8 would send the weight gradient to the SIMT engine (1.5 ms per call at batch 8, 256^2: the largest
            # single item of the train step).  Zero-padding the IMAGE to one 64-channel block puts it on the tcgen05
            # wgrad kernel instead (8x the flops, ~4x faster); the pad costs one 64-channel image write.
            x64 = torch.zeros(x.shape[:3] + (64,), device=x.device, dtype=x.dtype)
            x64[..., :8] = x
            dw64 = torch.zeros((m.shape[0], 64) + tuple(m.shape[2:]), device=m.device, dtype=torch.float32)
            ConvGeom("conv", 64, g.Cout, g.k, g.stride, g.pad, g.dil).wgrad(x64, dy, dw64, db, dy_c_off=dy_c_off)
            dw = dw64[:, :8].contiguous()
        else:
            g.wgrad(x, dy, dw, db, dy_c_off=dy_c_off,
                    scratch=G.scratch(dw.numel(), m.device) if sink is not None else None)
        if name == "initial.0":
            dw = dw[:, :3].contiguous()
        if name == "output.0":
            dw = dw[:3].contiguous()
            db = db[:3].contiguous() if db is not None else None
        if sink is not None:
            if not direct:
                sink[f"{name}.weight"].add_(dw)
                if db is not None:
                    sink[f"{name}.bias"].add_(db)
        else:
            if db is None:
                db = torch.zeros(nb if name != "output.0" else 3, device=m.device, dtype=torch.float32)
            G[f"{name}.weight"] = dw if f"{name}.weight" not in G else G[f"{name}.weight"] + dw
            G[f"{name}.bias"] = db if f"{name}.bias" not in G else G[f"{name}.bias"] + db
        if not need_dx:
            return None
        return g.dgrad(dy, self._packed(P, name, "dgrad", dtype), in_hw or x.shape[1:3], out=dx_out,
                       accumulate=accumulate, dy_c_off=dy_c_off)

    def _stage_bwd(self, P, G, s, sv, da2, dtype, A=None):
        if "y0" not in sv:  # checkpointed: recompute the stage from its input (enhanced_generator.py:186-208)
            _, sv = self._stage_fwd(P, s, sv["a_in"], dtype, keep=True, A=A)
        C = self.width[s]
        df = self._in_bwd(sv["f"], sv["stf"], da2, A, f"{s}.4.fusion.1")
        dbn = self._conv_bwd(P, G, f"{s}.4.fusion.0", sv["bn"], df, dtype)
        db = self._in_bwd(sv["b"], sv["stb"], dbn, A, f"{s}.4.branch")
        if self.use_slab and dtype == torch.bfloat16 and C in self._msb_dprog and db.shape[2] % 8 == 0:
            # data gradient of the four branches: one row-slab launch (N = C per tap) + the residual add
            wn = [f"{s}.4.branch{i}.0.weight" for i in range(1, 5)]
            dprog = self._msb_dprog[C]
            wsl = self._slab_cached(P, (s, "msb_dw"), wn, lambda: slab.msb_dgrad_weight_slab(dprog, [P[k].detach() for k in wn]))
            da1 = ops.add(slab.conv_slab(dprog, db, wsl, None), da2)
            for i in range(1, 5):
                self._conv_bwd(P, G, f"{s}.4.branch{i}.0", sv["a1"], db, dtype, dy_c_off=(i - 1) * (C // 4), need_dx=False)
        else:
            da1 = da2.clone()  # residual path: d(a1) starts as d(a2)
            for i in range(1, 5):
                self._conv_bwd(P, G, f"{s}.4.branch{i}.0", sv["a1"], db, dtype, dy_c_off=(i - 1) * (C // 4),
                               dx_out=da1, accumulate=True)
        datt = self._conv_bwd(P, G, f"{s}.3.proj", sv["att"], da1, dtype)
        dqkv = ops.local_attn_bwd(sv["qkv"], datt)
        da0 = self._conv_bwd(P, G, f"{s}.3.qkv", sv["a0"], dqkv, dtype)
        dy0 = self._in_bwd(sv["y0"], sv["st0"], da0, A, f"{s}.1")
        return self._conv_bwd(P, G, f"{s}.0", sv["a_in"], dy0, dtype)

    def grad_sink(self, sinks, device):
        """G argument of decode_bwd / encode_bwd that accumulates into `sinks` ({state_dict key: fp32 tensor})."""
        return GradSink(sinks, self._arena_floats, device)

    def grad_sink_done(self, G):
        self._arena_floats = max(self._arena_floats, G.used)

    def decode_bwd(self, P, G, saved, dy, dtype, A=None):
        """dy: fp32 NCHW grad of the image.  Returns d(a) at the decoder input (NHWC).  A: the forward's StyleAffine, its sums
        arena allocated (style_affine_begin_bwd)."""
        dz = ops.tanh_bwd_nchw(saved["y"], dy, dtype, self.edge_pad(dtype))
        da = self._conv_bwd(P, G, "output.0", saved["a_last"], dz, dtype)
        for s in ("up2", "up1"):
            da = self._stage_bwd(P, G, s, saved[s], da, dtype, A)
        return da

    def encode_bwd(self, P, G, saved, da, dtype, need_dx, A=None):
        for s in ("down2", "down1"):
            da = self._stage_bwd(P, G, s, saved[s], da, dtype, A)
        dyi = self._in_bwd(saved["yi"], saved["sti"], da, A, "initial.1")
        dx0 = self._conv_bwd(P, G, "initial.0", saved["x0"], dyi, dtype, need_dx=need_dx)
        if not need_dx:
            return None
        return ops.nhwc_to_nchw(dx0, 3)
