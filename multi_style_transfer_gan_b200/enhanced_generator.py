"""Drop-in replacement for the reference's ``enhanced_generator`` module
(reference: enhanced_generator.py).  Same class names, constructor signatures, module tree and
``state_dict`` keys; the computation runs on hand-written sm_100a kernels through the C-ABI in
include/msg_b200.h.  There is no CPU path: calling a model on CPU tensors (or without the built
extension) raises.

    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator, EnhancedDiscriminator

Precision: ``model.set_precision("fp32" | "bf16")`` (default "fp32" = the parity mode, <=1e-4 vs the
reference); inside ``torch.autocast("cuda")`` -- which is how the reference trains
(enhanced_train.py:61,88) -- the bf16 tensor-core path is used automatically.

Style-conditional generator (an extension, not in the reference): ``model.enable_style_affine(S)`` gives every
InstanceNorm an [S, C] affine (conditional instance norm, Dumoulin et al.) and ``model(x, style=w)`` blends the S
styles per image, gamma_n = sum_s w[n, s] gamma_s (beta alike), in one forward pass.
"""
import math

import torch
import torch.nn as nn

from . import _lib
from .discriminator_engine import D_CONVS, DiscriminatorEngine
from .generator_engine import GeneratorEngine

__all__ = ["LocalAttention", "MultiScaleBlock", "EnhancedGenerator", "EnhancedDiscriminator",
           "StructuralTransformerBlock"]


# ------------------------------------------------------------------------------------------------
# parameter holders (mirror the reference's module tree so that state_dict keys are identical)
# ------------------------------------------------------------------------------------------------
class _NoForward(nn.Module):
    def forward(self, *a, **k):
        raise RuntimeError(
            f"{type(self).__name__} only holds parameters; the computation is fused into the parent "
            "model's CUDA path (call the EnhancedGenerator / EnhancedDiscriminator itself)")


class Conv2d(_NoForward):
    """Holds weight [Cout,Cin,k,k] + bias like nn.Conv2d, with nn.Conv2d's default init (same RNG
    draws as the reference's constructor)."""
    transposed = False

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0, dilation=1):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding, self.dilation = kernel_size, stride, padding, dilation
        shape = self._weight_shape()
        self.weight = nn.Parameter(torch.empty(shape))
        self.bias = nn.Parameter(torch.empty(out_channels))
        self.reset_parameters()

    def _weight_shape(self):
        return (self.out_channels, self.in_channels, self.kernel_size, self.kernel_size)

    def reset_parameters(self):
        nn.init.kaiming_uniform_(self.weight, a=math.sqrt(5))
        fan_in, _ = nn.init._calculate_fan_in_and_fan_out(self.weight)
        bound = 1 / math.sqrt(fan_in) if fan_in > 0 else 0
        nn.init.uniform_(self.bias, -bound, bound)

    def extra_repr(self):
        return (f"{self.in_channels}, {self.out_channels}, kernel_size={self.kernel_size}, stride={self.stride}, "
                f"padding={self.padding}, dilation={self.dilation}")


class ConvTranspose2d(Conv2d):
    transposed = True

    def _weight_shape(self):
        return (self.in_channels, self.out_channels, self.kernel_size, self.kernel_size)


class InstanceNorm2d(_NoForward):
    """affine=False, track_running_stats=False, eps=1e-5: no parameters, no state_dict entries -- until
    EnhancedGenerator.enable_style_affine gives it weight / bias [S, C] (nn.InstanceNorm2d(affine=True) with a leading
    style axis, initialised to 1 and 0)."""

    def __init__(self, num_features):
        super().__init__()
        self.num_features, self.eps = num_features, 1e-5
        self.weight = None
        self.bias = None

    def _enable_style_affine(self, num_styles, device):
        self.weight = nn.Parameter(torch.ones(num_styles, self.num_features, device=device))
        self.bias = nn.Parameter(torch.zeros(num_styles, self.num_features, device=device))


class ReLU(_NoForward):
    pass


class LeakyReLU(_NoForward):
    def __init__(self, negative_slope=0.2):
        super().__init__()
        self.negative_slope = negative_slope


class Tanh(_NoForward):
    pass


class AdaptiveAvgPool2d(_NoForward):
    def __init__(self, output_size=1):
        super().__init__()
        self.output_size = output_size


class LocalAttention(_NoForward):
    """reference: enhanced_generator.py:6-47 (window_size is 4 everywhere on the path)."""

    def __init__(self, channels, window_size=8):
        super().__init__()
        self.window_size = window_size
        self.qkv = Conv2d(channels, channels * 3, 1)
        self.proj = Conv2d(channels, channels, 1)


class MultiScaleBlock(_NoForward):
    """reference: enhanced_generator.py:49-84."""

    def __init__(self, channels):
        super().__init__()
        q = channels // 4
        self.branch1 = nn.Sequential(Conv2d(channels, q, 1), InstanceNorm2d(q), ReLU())
        self.branch2 = nn.Sequential(Conv2d(channels, q, 3, padding=1, dilation=1), InstanceNorm2d(q), ReLU())
        self.branch3 = nn.Sequential(Conv2d(channels, q, 3, padding=2, dilation=2), InstanceNorm2d(q), ReLU())
        self.branch4 = nn.Sequential(Conv2d(channels, q, 3, padding=4, dilation=4), InstanceNorm2d(q), ReLU())
        self.fusion = nn.Sequential(Conv2d(channels, channels, 1), InstanceNorm2d(channels), ReLU())


class StructuralTransformerBlock(nn.Module):
    """The reference imports this class from a module that is NOT in its repository
    (enhanced_generator.py:4); only the interface is known: ctor (dim), call (x[B,HW/16,4c],
    style[B,4c], orig[B,3,H,W]) -> same shape as x.  This stand-in is the identity (parity
    unpinned, SURVEY.md F2).  Replace entries of ``model.transformer_blocks`` with real modules to
    plug an implementation in: they then run through stock PyTorch between down2 and up1."""

    def __init__(self, dim):
        super().__init__()
        self.dim = dim

    def forward(self, x, style, orig_input):
        return x


# ------------------------------------------------------------------------------------------------
# autograd glue
# ------------------------------------------------------------------------------------------------
def _resolve_dtype(precision):
    if torch.is_autocast_enabled():
        return torch.bfloat16
    return torch.bfloat16 if precision == "bf16" else torch.float32


def _check_input(x, what):
    if not isinstance(x, torch.Tensor) or x.dim() != 4:
        raise RuntimeError(f"{what}: expected a 4-D [B,3,H,W] tensor")
    if not x.is_cuda:
        raise _lib.MsgError(f"{what}: input is on {x.device}; this package has no CPU path "
                            "(the reference itself is the CPU implementation)")
    _lib.require_device(x.device.index)


# A (argument 4 of the functions below): the StyleAffine tables of a style-conditional forward, or None.  It is not a tensor
# input: no gradient flows to the style mix; the backward turns the per-image affine gradients into those of the [S, C]
# parameters itself (GeneratorEngine.style_affine_end_bwd).
class _GeneratorFn(torch.autograd.Function):
    """Whole-generator op: one autograd node, manual backward over saved NHWC activations."""

    @staticmethod
    def forward(ctx, model, dtype, keys, grad_on, A, x, *params):
        eng = model._engine
        P = dict(zip(keys, params))
        need = grad_on and (ctx.needs_input_grad[5] or any(ctx.needs_input_grad[6:]))   # needs_input_grad ignores no_grad
        save = ("ckpt" if model._checkpointing else "full") if need else False
        a, s_enc = eng.encode(P, x, dtype, save, A)
        y, s_dec = eng.decode(P, a, dtype, save, A)
        if need:
            ctx.model, ctx.dtype, ctx.keys, ctx.saved, ctx.A = model, dtype, keys, (s_enc, s_dec), A
            ctx.save_for_backward(*params)
        return y

    @staticmethod
    def backward(ctx, dy):
        eng, dtype, keys, A = ctx.model._engine, ctx.dtype, ctx.keys, ctx.A
        P = dict(zip(keys, ctx.saved_tensors))
        s_enc, s_dec = ctx.saved
        # the optimizer registered the views of its flat gradient buffer (EnhancedCycleGAN._build_optimizers): accumulate there
        # directly and hand autograd nothing to add
        sinks = getattr(ctx.model, "_grad_sinks", None)
        use_sink = sinks is not None and all(ctx.needs_input_grad[6:]) and all(k in sinks for k in keys)
        G = eng.grad_sink(sinks, dy.device) if use_sink else {}
        dy = dy.contiguous().float()
        if A is not None:
            eng.style_affine_begin_bwd(A)
        da = eng.decode_bwd(P, G, s_dec, dy, dtype, A)
        dx = eng.encode_bwd(P, G, s_enc, da, dtype, need_dx=ctx.needs_input_grad[5], A=A)
        if A is not None:
            eng.style_affine_end_bwd(G, A)
        ctx.saved = ctx.A = None
        if use_sink:
            eng.grad_sink_done(G)
            return (None, None, None, None, None, dx) + (None,) * len(keys)
        grads = tuple(G.get(k) if ctx.needs_input_grad[6 + i] else None for i, k in enumerate(keys))
        return (None, None, None, None, None, dx) + grads


class _EncoderFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, dtype, keys, grad_on, A, x, *params):
        eng = model._engine
        P = dict(zip(keys, params))
        need = grad_on and (ctx.needs_input_grad[5] or any(ctx.needs_input_grad[6:]))   # needs_input_grad ignores no_grad
        save = ("ckpt" if model._checkpointing else "full") if need else False
        a, s_enc = eng.encode(P, x, dtype, save, A)
        if need:
            ctx.model, ctx.dtype, ctx.keys, ctx.saved, ctx.A = model, dtype, keys, s_enc, A
            ctx.save_for_backward(*params)
        return a.float()  # [N,h,w,4c] tokens-major, fp32 for the user's blocks

    @staticmethod
    def backward(ctx, da):
        eng, dtype, keys, A = ctx.model._engine, ctx.dtype, ctx.keys, ctx.A
        P = dict(zip(keys, ctx.saved_tensors))
        G = {}
        if A is not None:
            eng.style_affine_begin_bwd(A)
        dx = eng.encode_bwd(P, G, ctx.saved, da.contiguous().to(dtype), dtype, need_dx=ctx.needs_input_grad[5], A=A)
        if A is not None:
            eng.style_affine_end_bwd(G, A)
        ctx.saved = ctx.A = None
        return (None, None, None, None, None, dx) + tuple(G.get(k) for k in keys)


class _DecoderFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, dtype, keys, grad_on, A, a, *params):
        eng = model._engine
        P = dict(zip(keys, params))
        need = grad_on and (ctx.needs_input_grad[5] or any(ctx.needs_input_grad[6:]))   # needs_input_grad ignores no_grad
        save = ("ckpt" if model._checkpointing else "full") if need else False
        y, s_dec = eng.decode(P, a.contiguous().to(dtype), dtype, save, A)
        if need:
            ctx.model, ctx.dtype, ctx.keys, ctx.saved, ctx.A = model, dtype, keys, s_dec, A
            ctx.save_for_backward(*params)
        return y

    @staticmethod
    def backward(ctx, dy):
        eng, dtype, keys, A = ctx.model._engine, ctx.dtype, ctx.keys, ctx.A
        P = dict(zip(keys, ctx.saved_tensors))
        G = {}
        if A is not None:
            eng.style_affine_begin_bwd(A)
        da = eng.decode_bwd(P, G, ctx.saved, dy.contiguous().float(), dtype, A)
        if A is not None:
            eng.style_affine_end_bwd(G, A)
        ctx.saved = ctx.A = None
        return (None, None, None, None, None, da.float()) + tuple(G.get(k) for k in keys)


class EnhancedGenerator(nn.Module):
    """reference: enhanced_generator.py:86-228."""

    def __init__(self, channels=64, num_transformer_blocks=3):
        super().__init__()
        c = channels
        self.initial = nn.Sequential(Conv2d(3, c, 7, 1, 3), InstanceNorm2d(c), ReLU())
        self.down1 = nn.Sequential(Conv2d(c, c * 2, 4, 2, 1), InstanceNorm2d(c * 2), ReLU(),
                                   LocalAttention(c * 2, window_size=4), MultiScaleBlock(c * 2))
        self.down2 = nn.Sequential(Conv2d(c * 2, c * 4, 4, 2, 1), InstanceNorm2d(c * 4), ReLU(),
                                   LocalAttention(c * 4, window_size=4), MultiScaleBlock(c * 4))
        self.transformer_blocks = nn.ModuleList(
            [StructuralTransformerBlock(dim=c * 4) for _ in range(num_transformer_blocks)])
        self.up1 = nn.Sequential(ConvTranspose2d(c * 4, c * 2, 4, 2, 1), InstanceNorm2d(c * 2), ReLU(),
                                 LocalAttention(c * 2, window_size=4), MultiScaleBlock(c * 2))
        self.up2 = nn.Sequential(ConvTranspose2d(c * 2, c, 4, 2, 1), InstanceNorm2d(c), ReLU(),
                                 LocalAttention(c, window_size=4), MultiScaleBlock(c))
        self.output = nn.Sequential(Conv2d(c, 3, 7, 1, 3), Tanh())
        self.style_encoder = nn.Sequential(AdaptiveAvgPool2d(1), nn.Flatten(), nn.Linear(c * 4, c * 4), nn.ReLU(True))
        self.apply(self._init_weights)
        self.channels = c
        self._engine = GeneratorEngine(c)
        self._checkpointing = False
        self.precision = "fp32"
        self.num_styles = None

    def _init_weights(self, m):
        # enhanced_generator.py:152-161 (fan_out of a ConvTranspose2d weight is size(0)*k*k -- the
        # reference's quirk is reproduced by torch's own fan computation)
        if isinstance(m, Conv2d):
            nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            nn.init.constant_(m.bias, 0)

    # ---- reference API -----------------------------------------------------------------------
    def gradient_checkpointing_enable(self):
        """reference: enhanced_generator.py:163-177.  Here: keep only each stage's input and
        recompute the stage inside backward (results unchanged up to fp32 summation order)."""
        for m in (self.down1, self.down2, self.transformer_blocks, self.up1, self.up2):
            m.requires_grad_(True)
        self.use_checkpointing = True
        self._checkpointing = True

    def param_version(self):
        """Identity + in-place version of every parameter (captured CUDA graphs are keyed on it)."""
        return tuple((q.data_ptr(), q._version) for q in self.parameters())

    def set_precision(self, precision):
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self.precision = precision
        return self

    def enable_style_affine(self, num_styles):
        """Makes the model style-conditional (conditional instance norm): each of the 25 InstanceNorm holders gets a weight and
        a bias Parameter [num_styles, C], initialised to 1 and 0 (no RNG draws), and ``forward`` then requires ``style``.
        The 70 plain state_dict keys keep their order; a plain checkpoint loads with strict=False (the 50 affine keys are
        then missing and keep their identity init).  Returns self."""
        S = int(num_styles)
        if S < 1:
            raise ValueError(f"num_styles must be >= 1, got {num_styles}")
        if self.num_styles is not None:
            raise ValueError(f"the model is already style-conditional ({self.num_styles} styles)")
        dev = self.initial[0].weight.device
        for name, _, holders in self._engine.sites:
            for h in holders:
                self.get_submodule(h)._enable_style_affine(S, dev)
        self.num_styles = S
        self._engine.invalidate()
        return self

    def _style_mix(self, style, x):
        """Validates ``style`` before any device work: [S] (one mix for the batch) or [B, S] (one per image), fp32, no grad.
        Returns it as a tensor (None for a plain model)."""
        S = self.num_styles
        if S is None:
            if style is not None:
                raise ValueError("style= needs a style-conditional model: call enable_style_affine(num_styles) first")
            return None
        if style is None:
            raise ValueError(f"this model is style-conditional ({S} styles): pass style= ([{S}] or [B, {S}] weights)")
        if isinstance(style, torch.Tensor):
            if style.requires_grad:
                raise ValueError("style must not require grad: gradients w.r.t. the style weights are not computed")
            if style.dtype != torch.float32:
                raise ValueError(f"style must be float32, got {style.dtype}")
            w = style
        else:
            w = torch.as_tensor(style, dtype=torch.float32)
        B = x.shape[0] if isinstance(x, torch.Tensor) and x.dim() == 4 else None
        if not ((w.dim() == 1 and w.shape[0] == S) or (w.dim() == 2 and tuple(w.shape) == (B, S))):
            raise ValueError(f"style must be [{S}] or [{B}, {S}], got {tuple(w.shape)}")
        return w

    def invalidate_packed_weights(self):
        """Call after mutating parameters through raw pointers (the fused Adam does)."""
        self._engine.invalidate()

    def _kernel_params(self):
        keys, params = [], []
        for k, p in self.named_parameters():
            if k.startswith("transformer_blocks.") or k.startswith("style_encoder."):
                continue
            keys.append(k)
            params.append(p)
        return tuple(keys), params

    def _blocks_are_identity(self):
        return all(type(b) is StructuralTransformerBlock for b in self.transformer_blocks)

    def forward(self, x, style=None):
        """style: the style mix of a conditional model (enable_style_affine), fp32 [S] or [B, S] on the host or the device,
        used as given (no normalisation); a plain model takes none."""
        w = self._style_mix(style, x)
        _check_input(x, "EnhancedGenerator")
        dtype = _resolve_dtype(self.precision)
        keys, params = self._kernel_params()
        xin = x if x.dtype == torch.float32 else x.float()
        # autograd.Function.forward always runs with grad mode off and ctx.needs_input_grad ignores no_grad, so the
        # caller's grad mode is recorded here: under no_grad nothing is saved and the inference schedule is used
        # (passed as an argument, not stored on the module: forward stays re-entrant across threads, gan_login_gui.py:755-767)
        grad_on = torch.is_grad_enabled()
        with torch.cuda.device(x.device):      # kernels launch on the tensors' device, whatever the caller's current device is
            A = None
            if w is not None:                  # the per-image affine tables of all 13 norm sites: one launch per call
                w = w.to(x.device).expand(x.shape[0], self.num_styles).contiguous()
                A = self._engine.style_tables(dict(zip(keys, params)), w)
            if self._blocks_are_identity():
                # style_encoder output is only consumed by the (identity) blocks: dead, skipped
                return _GeneratorFn.apply(self, dtype, keys, grad_on, A, xin.contiguous(), *params)
            a = _EncoderFn.apply(self, dtype, keys, grad_on, A, xin.contiguous(), *params)     # [B,h,w,4c]
            B, h, w, C = a.shape
            style = self.style_encoder[3](self.style_encoder[2](a.mean(dim=(1, 2))))  # :142-147, :216
            t = a.reshape(B, h * w, C)                                                # :218-219
            for block in self.transformer_blocks:
                t = block(t, style, x)                                                # :222-223
            return _DecoderFn.apply(self, dtype, keys, grad_on, A, t.reshape(B, h, w, C), *params)

    def load_state_dict(self, state_dict, strict=True, **kw):
        out = super().load_state_dict(state_dict, strict=strict, **kw)
        self._engine.invalidate()
        return out


# ------------------------------------------------------------------------------------------------
# discriminator
# ------------------------------------------------------------------------------------------------
class SpectralNormConv2d(_NoForward):
    """nn.Conv2d wrapped by the old-style torch.nn.utils.spectral_norm: parameters ``bias``,
    ``weight_orig`` and buffers ``weight_u``, ``weight_v`` (state_dict order of the reference)."""

    def __init__(self, in_channels, out_channels, kernel_size, stride=1, padding=0):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.kernel_size, self.stride, self.padding = kernel_size, stride, padding
        w = torch.empty(out_channels, in_channels, kernel_size, kernel_size)
        nn.init.kaiming_uniform_(w, a=math.sqrt(5))
        fan_in, _ = nn.init._calculate_fan_in_and_fan_out(w)
        bound = 1 / math.sqrt(fan_in)
        self.bias = nn.Parameter(torch.empty(out_channels))
        nn.init.uniform_(self.bias, -bound, bound)
        self._w_init = w

    def apply_spectral_norm(self):
        w = self._w_init
        del self._w_init
        h, wd = w.shape[0], w.numel() // w.shape[0]
        u = nn.functional.normalize(w.new_empty(h).normal_(0, 1), dim=0, eps=1e-12)
        v = nn.functional.normalize(w.new_empty(wd).normal_(0, 1), dim=0, eps=1e-12)
        self.weight_orig = nn.Parameter(w)
        self.register_buffer("weight_u", u)
        self.register_buffer("weight_v", v)


class _DiscriminatorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, dtype, training, keys, grad_on, x, *params):
        eng = model._engine
        P = dict(zip(keys, params))
        P.update(model._buffers_dict())
        need_dx = grad_on and ctx.needs_input_grad[5]
        need_dw = grad_on and any(ctx.needs_input_grad[6:])
        save = need_dx or need_dw
        ctx.set_materialize_grads(False)   # unused head (score or struct) -> None, not zeros
        score, struct, saved = eng.forward(P, x, dtype, training, save)
        if save:
            ctx.model, ctx.dtype, ctx.keys, ctx.saved = model, dtype, keys, saved
            ctx.need = (need_dx, need_dw)
            ctx.save_for_backward(*params)
        return score, struct

    @staticmethod
    def backward(ctx, dscore, dstruct):
        eng, dtype, keys = ctx.model._engine, ctx.dtype, ctx.keys
        P = dict(zip(keys, ctx.saved_tensors))
        need_dx, need_dw = ctx.need
        dx, G = eng.backward(P, ctx.saved, None if dscore is None else dscore.contiguous(),
                             None if dstruct is None else dstruct.contiguous(), dtype, need_dx, need_dw)
        ctx.saved = None
        grads = tuple(G.get(k) if ctx.needs_input_grad[6 + i] else None for i, k in enumerate(keys))
        return (None, None, None, None, None, dx) + grads


class EnhancedDiscriminator(nn.Module):
    """reference: enhanced_generator.py:230-275."""

    def __init__(self, channels=64):
        super().__init__()
        c = channels
        S = SpectralNormConv2d
        self.main = nn.Sequential(
            S(3, c, 4, 2, 1), LeakyReLU(0.2),
            S(c, c * 2, 4, 2, 1), InstanceNorm2d(c * 2), LeakyReLU(0.2),
            S(c * 2, c * 4, 4, 2, 1), InstanceNorm2d(c * 4), LeakyReLU(0.2),
            S(c * 4, c * 8, 4, 2, 1), InstanceNorm2d(c * 8), LeakyReLU(0.2))
        self.batch_head = nn.Sequential(S(c * 8, 1, 4, 1, 1), AdaptiveAvgPool2d(1))
        self.structure_head = nn.Sequential(S(c * 8, c * 8, 3, 1, 1), InstanceNorm2d(c * 8), LeakyReLU(0.2),
                                            S(c * 8, 1, 4, 1, 1))
        for m in self.modules():           # :269-271, same traversal order -> same RNG draws
            if isinstance(m, SpectralNormConv2d):
                m.apply_spectral_norm()
        self.channels = c
        self._engine = DiscriminatorEngine(c)
        self.precision = "fp32"

    def set_precision(self, precision):
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self.precision = precision
        return self

    def _buffers_dict(self):
        return {k: b for k, b in self.named_buffers()}

    def forward(self, x):
        _check_input(x, "EnhancedDiscriminator")
        dtype = _resolve_dtype(self.precision)
        keys, params = zip(*self.named_parameters())
        xin = x if x.dtype == torch.float32 else x.float()
        grad_on = torch.is_grad_enabled()    # see EnhancedGenerator.forward
        with torch.cuda.device(x.device):
            score, struct = _DiscriminatorFn.apply(self, dtype, self.training, tuple(keys), grad_on, xin.contiguous(), *params)
        return score.squeeze(), struct      # .squeeze(): 0-dim when B == 1 (:275)
