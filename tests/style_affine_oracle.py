"""CPU restatement (plain PyTorch) of the style-conditional EnhancedGenerator (EnhancedGenerator.enable_style_affine), the reference
the tests check the kernels against.  It is oracle.restate.generator_forward with every InstanceNorm followed by its per-image
affine, IN(x) * gamma_n + beta_n with gamma_n = w[n] @ gamma_s (beta alike) -- oracle.restate.blended_affine_instance_norm with
one mix per image.  The four branch norms of a MultiScaleBlock stay per branch, as in the module tree."""
import torch
import torch.nn.functional as F

from oracle.restate import blended_affine_instance_norm, instance_norm, local_attention

STAGES = ("down1", "down2", "up1", "up2")


def affine_norm(sd, w):
    """norm(x, holder) for a batch: w [B, S] (or [S], one mix for the batch)."""
    def norm(x, holder):
        ww = w if w.dim() == 2 else w.expand(x.shape[0], -1)
        g = ww @ sd[f"{holder}.weight"]
        b = ww @ sd[f"{holder}.bias"]
        return instance_norm(x) * g[:, :, None, None] + b[:, :, None, None]
    return norm


def blended_norm(sd, w_row):
    """norm(x, holder) of ONE image's mix w_row [S], through oracle.restate.blended_affine_instance_norm."""
    def norm(x, holder):
        return blended_affine_instance_norm(x, sd[f"{holder}.weight"], sd[f"{holder}.bias"], w_row)
    return norm


def _msb(x, sd, prefix, norm):
    outs = []
    for i, (pad, dil) in enumerate([(0, 1), (1, 1), (2, 2), (4, 4)], start=1):
        y = F.conv2d(x, sd[f"{prefix}.branch{i}.0.weight"], sd[f"{prefix}.branch{i}.0.bias"], padding=pad, dilation=dil)
        outs.append(torch.relu(norm(y, f"{prefix}.branch{i}.1")))
    f = F.conv2d(torch.cat(outs, dim=1), sd[f"{prefix}.fusion.0.weight"], sd[f"{prefix}.fusion.0.bias"])
    return torch.relu(norm(f, f"{prefix}.fusion.1")) + x


def _stage(x, sd, name, transposed, norm):
    w, b = sd[f"{name}.0.weight"], sd[f"{name}.0.bias"]
    x = F.conv_transpose2d(x, w, b, stride=2, padding=1) if transposed else F.conv2d(x, w, b, stride=2, padding=1)
    x = torch.relu(norm(x, f"{name}.1"))
    x = local_attention(x, sd[f"{name}.3.qkv.weight"], sd[f"{name}.3.qkv.bias"],
                        sd[f"{name}.3.proj.weight"], sd[f"{name}.3.proj.bias"], ws=4)
    return _msb(x, sd, f"{name}.4", norm)


def generator_forward(sd, x, style=None, blocks=None, norm=None):
    """The conditional generator's forward: sd holds the 50 affine keys ([S, C]), style is the mix [S] or [B, S].  `norm`
    replaces the normalisation (default affine_norm(sd, style))."""
    if x.shape[2] % 16 or x.shape[3] % 16:
        raise RuntimeError("EnhancedGenerator: H and W must be multiples of 16")
    norm = norm or affine_norm(sd, style)
    orig = x
    x = F.conv2d(x, sd["initial.0.weight"], sd["initial.0.bias"], padding=3)
    x = torch.relu(norm(x, "initial.1"))
    x = _stage(x, sd, "down1", False, norm)
    x = _stage(x, sd, "down2", False, norm)
    if blocks:
        sty = torch.relu(F.linear(x.mean(dim=(2, 3)), sd["style_encoder.2.weight"], sd["style_encoder.2.bias"]))
        B, C, H, W = x.shape
        t = x.flatten(2).transpose(1, 2)
        for blk in blocks:
            t = blk(t, sty, orig)
        x = t.transpose(1, 2).reshape(B, C, H, W)
    x = _stage(x, sd, "up1", True, norm)
    x = _stage(x, sd, "up2", True, norm)
    return torch.tanh(F.conv2d(x, sd["output.0.weight"], sd["output.0.bias"], padding=3))


def random_affines(sd, S, seed):
    """gamma_s ~ 1 + 0.2 N(0, 1), beta_s ~ 0.1 N(0, 1) for every affine key of sd (in place)."""
    g = torch.Generator().manual_seed(seed)
    for k in sorted(sd):
        if k.endswith(".1.weight") and sd[k].dim() == 2:
            sd[k] = 1 + 0.2 * torch.randn(sd[k].shape, generator=g)
            kb = k[:-len("weight")] + "bias"
            sd[kb] = 0.1 * torch.randn(sd[kb].shape, generator=g)
    return sd
