"""Drop-in for the reference's ``pretrain.Generator`` (pretrain.py:60-97) and its masked-L1 training step
(:150-166) on the msg_b200 kernels.

Architecture: 4 x [Conv2d 4x4 s2 p1 (+BatchNorm2d) + LeakyReLU(0.2)] -> 3 x [ConvTranspose2d 4x4 s2 p1 + BatchNorm2d
+ ReLU] -> ConvTranspose2d(c, 3) + Tanh.  Same module tree, ``state_dict`` keys (``encoder.{0,2,3,5,6,8,9}.*``,
``decoder.{0,1,3,4,6,7,9}.*`` incl. ``running_mean / running_var / num_batches_tracked``) and default PyTorch init
in the same RNG order as the reference, so a seeded construction is bit-identical.

Kernels: the same conv / convT engines as the EnhancedGenerator (tcgen05 where Cin % 64 == 0).  BatchNorm over
(N, H, W) of an NHWC tensor IS InstanceNorm of the [1, N*H, W, C] view, so it reuses the IN machinery: statistics come
from the conv epilogue (summed over the batch), the apply kernel carries gamma / beta through its per-style affine
path, and the backward is two kernels, msg_instnorm_bwd_reduce -> msg_instnorm_bwd_apply with the affine, whose
per-channel reductions (sum g, sum g*xhat) are exactly d(beta), d(gamma).  Running statistics follow torch.nn.BatchNorm2d
(momentum 0.1, unbiased variance for the running estimate).

Data-parallel training: convert with torch.nn.SyncBatchNorm.convert_sync_batchnorm and wrap in DistributedDataParallel.
In train mode each SyncBatchNorm whose process group has more than one rank all-reduces its batch sums and element count in
the forward and its (sum g, sum g*xhat) between the two backward kernels, so N ranks of B/N images compute the step of one
process on B images (DESIGN.md 6).  d(gamma), d(beta) stay the local sums, which DDP averages.  DDP waits for a gradient of
every parameter: the engine returns all of them, including the analytically-zero ones of the conv biases in front of a
BatchNorm.  Plain BatchNorm2d layers, eval mode and a group of one rank exchange nothing.
"""
import torch
import torch.distributed as dist
import torch.nn as nn

from . import ops
from .generator_engine import _pad_dim
from .losses import l1
from .ops import ACT_LRELU, ACT_RELU, ACT_TANH, ConvGeom

ENC = ((0, None), (2, 3), (5, 6), (8, 9))      # (conv index, BatchNorm index) inside `encoder`  (pretrain.py:65-77)
DEC = ((0, 1), (3, 4), (6, 7), (9, None))      # (convT index, BatchNorm index) inside `decoder` (pretrain.py:80-91)
BN_MOMENTUM = 0.1                              # eps 1e-5 is the IN kernels' (kInEps, csrc/common.cuh)


def _edge_pad(dtype):
    return 4 if dtype == torch.float32 else 8


def bn_batch_stats(st, M, rm, rv, nbt, group=None):
    """Train-mode statistics of one BatchNorm layer, and the torch.nn.BatchNorm2d running-statistics update (momentum 0.1,
    unbiased variance).  Pure torch, no kernel: st holds the conv epilogue's per-image fp64 sums [N, C, 2] = (sum x,
    sum x^2) over this rank's M = N*H*W elements.

    group: None for a plain BatchNorm.  Otherwise the process group of a SyncBatchNorm: the batch sums and the element
    count, [2*C + 1] fp64, are summed over it by one all-reduce, the running statistics follow the global mean and the
    unbiased global variance (identical on every rank), and the returned sums are the global sums scaled by M / M_global,
    the local count the kernels normalise by (include/msg_b200.h).

    Returns (sums [1, C, 2] fp64, M / M_global as a 0-dim fp64 tensor, or None without a group)."""
    C = st.shape[1]
    stb = st.sum(0, keepdim=True)
    if group is None:
        Mg, unbias, scale = M, M / max(M - 1, 1), None
    else:
        buf = torch.cat([stb.reshape(-1), stb.new_full((1,), float(M))])
        dist.all_reduce(buf, group=group)
        stb, Mg = buf[:-1].view(1, C, 2), buf[-1]
        unbias, scale = Mg / (Mg - 1).clamp_min(1.0), M / Mg
    with torch.no_grad():
        mean = stb[0, :, 0] / Mg
        var = (stb[0, :, 1] / Mg - mean * mean).clamp_min(0.0)
        rm.mul_(1 - BN_MOMENTUM).add_((BN_MOMENTUM * mean).to(rm.dtype))
        rv.mul_(1 - BN_MOMENTUM).add_((BN_MOMENTUM * var * unbias).to(rv.dtype))
        nbt.add_(1)
    if scale is not None:
        stb = stb * scale
    return stb.contiguous(), scale


def bn_sync_groups(model):
    """BatchNorm name -> the process group its batch statistics are reduced over: the ``SyncBatchNorm`` layers of a
    model whose group (``process_group``, None meaning WORLD) has more than one rank.  Plain BatchNorm2d layers, and every
    layer when torch.distributed is not initialised, are absent: they normalise over the local batch."""
    if not (dist.is_available() and dist.is_initialized()):
        return {}
    out = {}
    for name, m in model.named_modules():
        if isinstance(m, nn.SyncBatchNorm):
            group = m.process_group if m.process_group is not None else dist.group.WORLD
            if dist.get_world_size(group) > 1:
                out[name] = group
    return out


class _Engine:
    """Forward / backward schedule of the BatchNorm auto-encoder over NHWC activations."""

    def __init__(self, c):
        self.c = c
        self.widths_enc = [(3, c), (c, 2 * c), (2 * c, 4 * c), (4 * c, 8 * c)]
        self.widths_dec = [(8 * c, 4 * c), (4 * c, 2 * c), (2 * c, c), (c, 3)]

    # ---- BatchNorm = InstanceNorm of the [1, N*H, W, C] view -------------------------------------------
    @staticmethod
    def _bn_fwd(y, st, gamma, beta, rm, rv, nbt, act, training, group):
        N, H, W, C = y.shape
        M = N * H * W
        scale = None
        if training:
            stb, scale = bn_batch_stats(st, M, rm, rv, nbt, group)
        else:
            stb = torch.empty((1, C, 2), device=y.device, dtype=torch.float64)
            stb[0, :, 0] = rm.double() * M
            stb[0, :, 1] = (rv.double() + rm.double() ** 2) * M
        one = torch.ones(1, device=y.device, dtype=torch.float32)
        out = ops.instnorm_apply(y.view(1, N * H, W, C), stb, act, gammas=gamma.detach().float().view(1, C).contiguous(),
                                 betas=beta.detach().float().view(1, C).contiguous(), w=one)
        return out.view(N, H, W, C), stb, scale

    @staticmethod
    def _bn_bwd(y, stb, da_out, gamma, beta, act, group, scale):
        """y: pre-norm conv output, da_out: gradient of act(gamma * xhat + beta).  reduce -> [all-reduce] -> apply.
        Returns (d y, d gamma, d beta); d gamma and d beta are this rank's sums, taken before the all-reduce: DDP averages
        them like every other parameter gradient (as torch.nn.SyncBatchNorm does)."""
        N, H, W, C = y.shape
        x, g = y.view(1, N * H, W, C), da_out.view(1, N * H, W, C)
        gam, bet = gamma.detach().float().contiguous(), beta.detach().float().contiguous()
        sums = ops.instnorm_bwd_reduce(x, stb, g, act, gam, bet)                    # (sum g, sum g * xhat)
        dbeta, dgamma = sums[0, :, 0].float(), sums[0, :, 1].float()
        if group is not None:
            dist.all_reduce(sums, group=group)
            sums.mul_(scale)                                                        # normalised to the local count
        dy = ops.instnorm_bwd_apply(x, stb, g, sums, act, gam, bet)
        return dy.view(N, H, W, C), dgamma, dbeta

    # ---- forward -----------------------------------------------------------------------------------------
    def forward(self, P, B, x, dtype, training, save, groups):
        """groups: bn_sync_groups of the model (train mode only)."""
        pad = _edge_pad(dtype)
        a = ops.nchw_to_nhwc(x, dtype, pad)
        tape = []
        for li, (ci, bi) in enumerate(ENC):
            cin, cout = self.widths_enc[li]
            w = P[f"encoder.{ci}.weight"].detach()
            if li == 0:
                w, cin = _pad_dim(w, 1, pad), pad
            g = ConvGeom("conv", cin, cout, 4, 2, 1)
            wp = g.pack_fwd(w.float().contiguous(), dtype)
            bias = P[f"encoder.{ci}.bias"].detach().float().contiguous()
            if bi is None:
                y = g.forward(a, wp, bias, act=ACT_LRELU)
                tape.append(("conv_act", f"encoder.{ci}", None, g, w, a, y, None, y, ACT_LRELU))
                a = y
            else:
                st = ops.new_stats(a.shape[0], cout, a.device)
                y = g.forward(a, wp, bias, stats=st)
                pre = f"encoder.{bi}"
                an, stb, scale = self._bn_fwd(y, st, P[pre + ".weight"], P[pre + ".bias"], B[pre + ".running_mean"],
                                              B[pre + ".running_var"], B[pre + ".num_batches_tracked"], ACT_LRELU, training,
                                              groups.get(pre))
                tape.append(("conv_bn", f"encoder.{ci}", pre, g, w, a, y, (stb, groups.get(pre), scale), an, ACT_LRELU))
                a = an
        out = None
        for li, (ci, bi) in enumerate(DEC):
            cin, cout = self.widths_dec[li]
            w = P[f"decoder.{ci}.weight"].detach()
            bias = P[f"decoder.{ci}.bias"].detach().float()
            if bi is None:
                w, bias, cout = _pad_dim(w, 1, pad), _pad_dim(bias, 0, pad), pad
            g = ConvGeom("convT", cin, cout, 4, 2, 1)
            wp = g.pack_fwd(w.float().contiguous(), dtype)
            bias = bias.contiguous()
            if bi is None:
                N, H, W, _ = a.shape
                out = torch.empty((N, cout, 2 * H, 2 * W), device=a.device, dtype=torch.float32)
                g.forward(a, wp, bias, act=ACT_TANH, nchw_out=out)
                tape.append(("convT_tanh", f"decoder.{ci}", None, g, w, a, None, None, out, ACT_TANH))
            else:
                st = ops.new_stats(a.shape[0], cout, a.device)
                y = g.forward(a, wp, bias, stats=st)
                pre = f"decoder.{bi}"
                an, stb, scale = self._bn_fwd(y, st, P[pre + ".weight"], P[pre + ".bias"], B[pre + ".running_mean"],
                                              B[pre + ".running_var"], B[pre + ".num_batches_tracked"], ACT_RELU, training,
                                              groups.get(pre))
                tape.append(("convT_bn", f"decoder.{ci}", pre, g, w, a, y, (stb, groups.get(pre), scale), an, ACT_RELU))
                a = an
        return out[:, :3].contiguous(), (tape if save else None), out

    # ---- backward ----------------------------------------------------------------------------------------
    def backward(self, P, tape, y_full, dy, dtype, need_dx):
        pad = _edge_pad(dtype)
        G = {}
        d = ops.tanh_bwd_nchw(y_full[:, :3].contiguous(), dy.float().contiguous(), dtype, pad)   # [N, H, W, pad]
        for kind, cname, bname, g, w, a_in, y, bn, a_out, act in reversed(tape):
            if kind in ("conv_bn", "convT_bn"):
                d, dgamma, dbeta = self._bn_bwd(y, bn[0], d, P[bname + ".weight"], P[bname + ".bias"], act, bn[1], bn[2])
                G[bname + ".weight"], G[bname + ".bias"] = dgamma, dbeta
            elif kind == "conv_act":
                d = ops.act_bwd(a_out, d, act)
            dw = torch.zeros(tuple(w.shape), device=d.device, dtype=torch.float32)
            db = torch.zeros(g.Cout, device=d.device, dtype=torch.float32)
            g.wgrad(a_in, d, dw, db)
            if cname == "encoder.0":
                dw = dw[:, :3].contiguous()
            if cname == "decoder.9":
                dw, db = dw[:, :3].contiguous(), db[:3].contiguous()
            G[cname + ".weight"], G[cname + ".bias"] = dw, db
            if cname == "encoder.0" and not need_dx:
                return G, None
            d = g.dgrad(d, g.pack_dgrad(w.float().contiguous(), dtype), a_in.shape[1:3])
        return G, ops.nhwc_to_nchw(d, 3)


class _PretrainFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, model, dtype, training, keys, grad_on, x, *params):
        P = dict(zip(keys, params))
        need = grad_on and (ctx.needs_input_grad[5] or any(ctx.needs_input_grad[6:]))
        if need and not training:
            raise NotImplementedError("pretrain.Generator (msg_b200): backward is implemented for train() mode "
                                      "(batch statistics); use no_grad for eval-mode inference")
        groups = bn_sync_groups(model) if training else {}
        y, tape, y_full = model._engine.forward(P, dict(model.named_buffers()), x, dtype, training, need, groups)
        if need:
            ctx.model, ctx.dtype, ctx.keys, ctx.tape, ctx.y_full = model, dtype, keys, tape, y_full
            ctx.save_for_backward(*params)
        return y

    @staticmethod
    def backward(ctx, dy):
        P = dict(zip(ctx.keys, ctx.saved_tensors))
        G, dx = ctx.model._engine.backward(P, ctx.tape, ctx.y_full, dy, ctx.dtype, ctx.needs_input_grad[5])
        ctx.tape = ctx.y_full = None
        grads = tuple(G.get(k) if ctx.needs_input_grad[6 + i] else None for i, k in enumerate(ctx.keys))
        return (None, None, None, None, None, dx) + grads


class Generator(nn.Module):
    """reference: pretrain.py:60-97 (same constructor, module tree and state_dict)."""

    def __init__(self, channels=64):
        super().__init__()
        c = channels
        self.encoder = nn.Sequential(
            nn.Conv2d(3, c, 4, 2, 1), nn.LeakyReLU(0.2),
            nn.Conv2d(c, c * 2, 4, 2, 1), nn.BatchNorm2d(c * 2), nn.LeakyReLU(0.2),
            nn.Conv2d(c * 2, c * 4, 4, 2, 1), nn.BatchNorm2d(c * 4), nn.LeakyReLU(0.2),
            nn.Conv2d(c * 4, c * 8, 4, 2, 1), nn.BatchNorm2d(c * 8), nn.LeakyReLU(0.2))
        self.decoder = nn.Sequential(
            nn.ConvTranspose2d(c * 8, c * 4, 4, 2, 1), nn.BatchNorm2d(c * 4), nn.ReLU(),
            nn.ConvTranspose2d(c * 4, c * 2, 4, 2, 1), nn.BatchNorm2d(c * 2), nn.ReLU(),
            nn.ConvTranspose2d(c * 2, c, 4, 2, 1), nn.BatchNorm2d(c), nn.ReLU(),
            nn.ConvTranspose2d(c, 3, 4, 2, 1), nn.Tanh())
        self.channels = c
        self._engine = _Engine(c)
        self.precision = "fp32"

    def set_precision(self, precision):
        if precision not in ("fp32", "bf16"):
            raise ValueError("precision must be 'fp32' or 'bf16'")
        self.precision = precision
        return self

    def forward(self, x):
        if x.dim() != 4 or x.shape[1] != 3:
            raise RuntimeError(f"pretrain.Generator expects [B,3,H,W], got {tuple(x.shape)}")
        if x.shape[2] % 16 or x.shape[3] % 16:
            raise RuntimeError(f"pretrain.Generator: H and W must be multiples of 16 (four stride-2 stages), got "
                               f"{x.shape[2]}x{x.shape[3]}")
        if not x.is_cuda:
            raise RuntimeError("pretrain.Generator (msg_b200): a CUDA tensor is required; there is no CPU path")
        dtype = torch.bfloat16 if (self.precision == "bf16" or torch.is_autocast_enabled()) else torch.float32
        keys, params = zip(*self.named_parameters())
        grad_on = torch.is_grad_enabled()      # an argument, not module state: forward stays re-entrant
        with torch.cuda.device(x.device):
            return _PretrainFn.apply(self, dtype, self.training, tuple(keys), grad_on, x.float().contiguous(), *params)


def set_seed(seed=42):
    """reference: pretrain.py:13-17 (host utility kept so `from pretrain import set_seed` resolves against dropin/)."""
    import random

    import numpy as np
    random.seed(seed)
    np.random.seed(seed)
    torch.manual_seed(seed)
    torch.cuda.manual_seed_all(seed)


class MonetPhotoDataset(torch.utils.data.Dataset):
    """reference: pretrain.py:20-57 -- `<root>/<split><domain>/*.jpg|*.png`, resize + centre crop to img_size,
    Normalize(0.5, 0.5), and an 8 x 8 grid mask hiding each cell with probability 0.4; returns
    (masked_image, image, mask).  Host-side data loading only (SURVEY.md section 2: not on the hot path); kept so that
    the reference's `from pretrain import MonetPhotoDataset` (enhanced_train.py:11, m_test.py:12) works with dropin/."""

    def __init__(self, root_dir, domain, split="train", img_size=256):
        from pathlib import Path

        from torchvision import transforms
        self.root_dir, self.domain, self.split, self.img_size = Path(root_dir), domain, split, img_size
        folder = self.root_dir / f"{split}{domain}"
        self.image_paths = list(folder.glob("*.jpg")) + list(folder.glob("*.png"))
        self.transform = transforms.Compose([
            transforms.Resize(img_size), transforms.CenterCrop(img_size), transforms.ToTensor(),
            transforms.Normalize((0.5, 0.5, 0.5), (0.5, 0.5, 0.5))])

    def __len__(self):
        return len(self.image_paths)

    def __getitem__(self, idx):
        import random

        from PIL import Image
        image = self.transform(Image.open(self.image_paths[idx]).convert("RGB"))
        mask = torch.ones_like(image)
        cell = self.img_size // 8
        for i in range(8):                 # same draw order as the reference: row-major cells, one random() each
            for j in range(8):
                if random.random() < 0.4:
                    mask[:, i * cell:(i + 1) * cell, j * cell:(j + 1) * cell] = 0
        return image * mask, image, mask


def pretrain_step(generator, optimizer, masked_imgs, real_imgs, masks, max_norm=1.0):
    """One optimisation step of pretrain.py:150-166: masked-L1 reconstruction loss on the hidden region, gradient-norm
    clipping at 1.0, optimizer step.  Returns the loss value (float)."""
    optimizer.zero_grad()
    generated = generator(masked_imgs)
    inv = 1 - masks
    loss = l1(generated * inv, real_imgs * inv)
    loss.backward()
    torch.nn.utils.clip_grad_norm_(generator.parameters(), max_norm=max_norm)
    optimizer.step()
    return float(loss.detach())
