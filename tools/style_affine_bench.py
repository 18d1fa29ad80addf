"""Style-conditional generator (EnhancedGenerator.enable_style_affine) against the plain one, on the device.

    python tools/style_affine_bench.py [--size 512] [--batch 32] [--iters 10] [--out result.json]

At c = 64, bf16, one micro-batch of `batch` images of size x size (inputs on the device, fp32 output):
  1. one plain forward vs one conditional forward (style = [0.2, 0.3, 0.5]): the cost of the affine;
  2. a three-style blend [0.2, 0.3, 0.5] in images/s: three plain generators + blend_outputs (MultiStyleStylizer) vs one
     conditional generator with style = [0.2, 0.3, 0.5] (MultiStyleStylizer with style=).
Timed with CUDA events around `iters` calls after warm-up; the card's name and power limit are read in the same run.
"""
import argparse
import copy
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator  # noqa: E402
from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name()


def timed(fn, iters, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(iters):
        fn()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("style_affine_bench: needs a CUDA device")
    dev = "cuda"
    mix = [0.2, 0.3, 0.5]
    gens = []
    for s in range(3):
        torch.manual_seed(s)
        gens.append(EnhancedGenerator(64, 0).to(dev).eval().set_precision("bf16"))
    Gc = copy.deepcopy(gens[0]).enable_style_affine(3)
    with torch.no_grad():           # three styles' affines: a plausible spread around the identity
        g = torch.Generator(device=dev).manual_seed(7)
        for n, p in Gc.named_parameters():
            if p.dim() == 2 and n.endswith(".1.weight"):
                p.copy_(1 + 0.2 * torch.randn(p.shape, generator=g, device=dev))
            elif p.dim() == 2 and n.endswith(".1.bias"):
                p.copy_(0.1 * torch.randn(p.shape, generator=g, device=dev))
    x = torch.rand(a.batch, 3, a.size, a.size, device=dev, generator=torch.Generator(device=dev).manual_seed(1)) * 2 - 1
    w = torch.tensor(mix, device=dev)
    res = {"card": card(), "size": a.size, "batch": a.batch, "channels": 64, "precision": "bf16", "iters": a.iters}
    with torch.no_grad():
        res["plain_forward_ms"] = timed(lambda: gens[0](x), a.iters)
        res["conditional_forward_ms"] = timed(lambda: Gc(x, style=w), a.iters)
        three = MultiStyleStylizer(gens, precision="bf16", micro_batch=a.batch)
        one = MultiStyleStylizer([Gc], precision="bf16", micro_batch=a.batch)
        t3 = timed(lambda: three(x, mix), a.iters)
        t1 = timed(lambda: one(x, [1.0], style=w), a.iters)
    res["three_generators_blend_ms"] = t3
    res["conditional_blend_ms"] = t1
    res["three_generators_blend_images_per_s"] = a.batch * 1e3 / t3
    res["conditional_blend_images_per_s"] = a.batch * 1e3 / t1
    res["blend_speedup"] = t3 / t1
    res["forward_ratio_conditional_over_plain"] = res["conditional_forward_ms"] / res["plain_forward_ms"]
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
