"""Times the per-pixel blend against the global blend at B = 32, 512x512, S = 3 styles, C = 3 (fp32 NCHW), inputs far larger
than the 126 MB L2 (3 styles + x + out = 5 x 100 MB), CUDA events around many launches:
  - msg_blend_outputs with global weights and the input term;
  - msg_blend_maps with [1, S+1, 1, 1], [B, S+1, 64, 64] and [B, S+1, 512, 512] maps, fp32 and uint8 output;
  - msg_gaussian_blur at sigma 8 on [B, S+1, 128, 128];
then the stylizer's images/s (c = 64, 3 blocks, bf16) with global weights and with [B, S+1, 64, 64] maps, alternating.
GB/s counts the bytes the algorithm must move: S + 1 input planes read, one plane written (4 B fp32 / 1 B uint8), plus the
map bytes.  Usage: python tools/blend_maps_bench.py [--reps R] [--stylizer-batch B] [--skip-stylizer]"""
import argparse
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_style_transfer_gan_b200 import ops  # noqa: E402


def timed(fn, reps):
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3   # us


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "nvidia-smi unavailable"
    return f"{torch.cuda.get_device_name()} ({q})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--stylizer-batch", type=int, default=32)
    ap.add_argument("--stylizer-rounds", type=int, default=3)
    ap.add_argument("--skip-stylizer", action="store_true")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("blend_maps_bench: needs a CUDA device")
    print(f"device: {card()}")
    B, C, H, W, S = 32, 3, 512, 512, 3
    g = torch.Generator(device="cuda").manual_seed(0)
    ys = [torch.rand(B, C, H, W, device="cuda", generator=g) * 2 - 1 for _ in range(S)]
    x = torch.rand(B, C, H, W, device="cuda", generator=g) * 2 - 1
    out = torch.empty_like(x)
    u8 = torch.empty(x.shape, device="cuda", dtype=torch.uint8)
    plane = B * C * H * W
    w = [0.2, 0.3, 0.5]

    def report(name, us, out_bytes, map_bytes=0):
        nbytes = (S + 1) * plane * 4 + plane * out_bytes + map_bytes
        print(f"{name:<52s} {us:9.1f} us  {nbytes / us / 1e3:7.1f} GB/s")
        return us

    base = report("blend_outputs  global w + w_x, fp32 out", timed(
        lambda: ops.blend_outputs(ys, w, x=x, w_x=0.25, out=out), args.reps), 4)
    report("blend_outputs  global w + w_x, uint8 out", timed(
        lambda: ops.blend_outputs(ys, w, x=x, w_x=0.25, out=u8), args.reps), 1)
    for shape in ((1, S + 1, 1, 1), (B, S + 1, 64, 64), (B, S + 1, H, W)):
        m = torch.rand(*shape, device="cuda", generator=g)
        mb = m.numel() * 4
        t = report(f"blend_maps     {list(shape)}, fp32 out", timed(lambda: ops.blend_maps(ys, m, x=x, out=out), args.reps), 4, mb)
        report(f"blend_maps     {list(shape)}, uint8 out", timed(lambda: ops.blend_maps(ys, m, x=x, out=u8), args.reps), 1, mb)
        print(f"{'':<52s} fp32: {t / base:.2f}x the global blend")
    m = torch.rand(B, S + 1, 128, 128, device="cuda", generator=g)
    us = timed(lambda: ops.gaussian_blur(m, 8.0), args.reps)
    print(f"{'gaussian_blur  sigma 8, ' + str(list(m.shape)):<52s} {us:9.1f} us  "
          f"{4 * m.numel() * 4 / us / 1e3:7.1f} GB/s (2 passes, read + write each)")
    del ys, x, out, u8

    if args.skip_stylizer:
        return
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    gens = []
    for s in range(S):
        torch.manual_seed(s)
        gens.append(EnhancedGenerator(channels=64, num_transformer_blocks=3).cuda())
    st = MultiStyleStylizer(gens, precision="bf16", micro_batch=32)
    nb = args.stylizer_batch
    xs = torch.rand(nb, 3, H, W, device="cuda", generator=g) * 2 - 1
    maps = torch.rand(nb, S + 1, 64, 64, device="cuda", generator=g)
    runs = {"global weights": lambda: st(xs, w, w_x=0.25), "[B, S+1, 64, 64] maps": lambda: st(xs, weight_maps=maps)}
    for fn in runs.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    for _ in range(args.stylizer_rounds):
        for k, fn in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[k].append(time.perf_counter() - t0)
    for k, ts in times.items():
        print(f"stylizer {k:<24s} " + "  ".join(f"{nb / t:7.1f}" for t in ts) + " images/s")


if __name__ == "__main__":
    main()
