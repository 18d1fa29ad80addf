"""CPU restatement (plain PyTorch) of the per-pixel blend (msg_blend_maps) and map feathering (msg_gaussian_blur), the
reference the tests check those kernels against.  enhanced_local_style.py:126-176 builds a per-region blend-ratio map,
smooths it with a Gaussian and blends per pixel as y*m + x*(1-m) (:232-236); this generalises that blend to S styles plus
the input image.  The blend arithmetic is oracle.restate.blend_outputs' with per-pixel weights, so constant maps reproduce
it exactly."""
import torch


def sample_maps(maps, H, W):
    """Weight maps [Bm,K,h,w] -> [Bm,K,H,W]: F.interpolate(mode="bilinear", align_corners=False)'s source indices, interpolated
    as a + t*(b - a), rows first, then columns (a constant map comes back exactly; F.interpolate is off by up to 1.2e-7)."""
    maps = maps.float()
    h, w = maps.shape[-2:]

    def index(n_out, n_in):
        scale = torch.tensor(float(n_in) / float(n_out), dtype=torch.float32)
        src = (scale * (torch.arange(n_out, dtype=torch.float32) + 0.5) - 0.5).clamp(min=0)
        i0 = src.to(torch.int64)
        return i0, (i0 + 1).clamp(max=n_in - 1), src - i0.to(torch.float32)

    r0, r1, ty = index(H, h)
    c0, c1, tx = index(W, w)
    top, bot = maps[..., r0, :], maps[..., r1, :]                     # [Bm,K,H,w]
    ty = ty[:, None]
    left = top[..., c0] + ty * (bot[..., c0] - top[..., c0])
    right = top[..., c1] + ty * (bot[..., c1] - top[..., c1])
    return left + tx * (right - left)


def gaussian_blur(planes, sigma):
    """scipy.ndimage.gaussian_filter(plane, sigma, mode="reflect", truncate=4.0) of every trailing [h, w] plane, in float64:
    radius int(4 sigma + 0.5), taps exp(-x^2 / 2 sigma^2) / sum, vertical then horizontal pass, half-sample-symmetric
    reflection of out-of-range indices (also when the radius exceeds the plane)."""
    x = planes.double()
    r = int(4.0 * float(sigma) + 0.5)
    if r == 0:
        return x.clone()
    d = torch.arange(-r, r + 1, dtype=torch.float64)
    taps = torch.exp(-0.5 * d * d / (float(sigma) ** 2))
    taps = taps / taps.sum()

    def fold(idx, n):
        idx = idx % (2 * n)
        return torch.where(idx >= n, 2 * n - 1 - idx, idx)

    def one_axis(t, dim):
        n = t.shape[dim]
        pos = torch.arange(n)
        out = torch.zeros_like(t)
        for k in range(2 * r + 1):
            out = out + taps[k] * t.index_select(dim, fold(pos + k - r, n))
        return out

    return one_axis(one_axis(x, x.dim() - 2), x.dim() - 1)


def blend_maps(ys, maps, x=None, gain=1.0, clip=None, normalize=False):
    """m = sample_maps(maps) [Bm,K,H,W] (K in {S, S+1}; map S weights x), optionally normalised to sum 1 per pixel (0 where
    the sum is 0), then oracle.restate.blend_outputs' arithmetic with per-pixel weights."""
    S = len(ys)
    m = sample_maps(maps, *ys[0].shape[-2:])
    if normalize:
        tot = m.sum(dim=1, keepdim=True)
        m = torch.where(tot != 0, m / torch.where(tot != 0, tot, torch.ones_like(tot)), torch.zeros_like(m))
    out = sum(m[:, s:s + 1] * ys[s] for s in range(S))
    if m.shape[1] == S + 1:
        out = out + m[:, S:S + 1] * x
    out = out * gain
    if clip is not None:
        out = out.clamp(*clip)
    return out
