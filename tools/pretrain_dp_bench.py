"""Data-parallel pretraining of pretrain.Generator(64) with synchronised BatchNorm: bf16, 256 x 256, 16 images per GPU,
FusedAdam, the model converted with torch.nn.SyncBatchNorm.convert_sync_batchnorm.
  - pretrain_step steps/s at world 1, and at world 2 over NCCL (DistributedDataParallel) when two GPUs are present;
  - at world 2, the time of the twelve statistics all-reduces of a step (CUDA events around each call on the compute
    stream, in a separate instrumented pass);
  - the BatchNorm backward of each of the six layers, the split reduce / apply kernels against the composition they
    replaced (act_bwd -> instnorm_bwd -> a second apply multiplying by gamma), alternating, CUDA events over many launches.
No tensor of the six BatchNorm shapes exceeds 33.5 MB in bf16, so these layer timings run largely from the 126 MB L2.
Usage: python tools/pretrain_dp_bench.py [--steps K] [--warmup W] [--reps R]"""
import argparse
import json
import os
import socket
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from multi_style_transfer_gan_b200 import ops  # noqa: E402

C, RES, PER_GPU = 64, 256, 16


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i",
                            str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        q = "nvidia-smi unavailable"
    return f"{torch.cuda.get_device_name()} ({q})"


def data(dev, seed):
    g = torch.Generator().manual_seed(seed)
    real = torch.rand(PER_GPU, 3, RES, RES, generator=g) * 2 - 1
    mask = (torch.rand(PER_GPU, 1, RES, RES, generator=g) > 0.4).float().expand(PER_GPU, 3, RES, RES).contiguous()
    return (real * mask).to(dev), real.to(dev), mask.to(dev)


def model(dev):
    from multi_style_transfer_gan_b200.enhanced_train import FusedAdam
    from multi_style_transfer_gan_b200.pretrain import Generator
    torch.manual_seed(0)
    G = torch.nn.SyncBatchNorm.convert_sync_batchnorm(Generator(C)).to(dev).set_precision("bf16").train()
    return G, FusedAdam(G.parameters(), lr=2e-4, betas=(0.5, 0.999))


def steps_per_s(D, opt, batch, steps, warmup):
    from multi_style_transfer_gan_b200.pretrain import pretrain_step
    for _ in range(warmup):
        pretrain_step(D, opt, *batch)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        pretrain_step(D, opt, *batch)
    torch.cuda.synchronize()
    return steps / (time.perf_counter() - t0)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank(rank, world, port, steps, warmup, q):
    import torch.distributed as dist
    from torch.nn.parallel import DistributedDataParallel as DDP

    from multi_style_transfer_gan_b200.pretrain import pretrain_step
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    G, opt = model(dev)
    D = DDP(G, device_ids=[rank])
    batch = data(dev, 100 + rank)
    sps = steps_per_s(D, opt, batch, steps, warmup)
    # instrumented pass: events on the compute stream around each statistics all-reduce (the call returns once the
    # stream waits for the collective)
    events, real_all_reduce = [], dist.all_reduce

    def timed_all_reduce(*a, **k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        r = real_all_reduce(*a, **k)
        e1.record()
        events.append((e0, e1))
        return r
    dist.all_reduce = timed_all_reduce
    try:
        for _ in range(steps):
            pretrain_step(D, opt, *batch)
    finally:
        dist.all_reduce = real_all_reduce
    torch.cuda.synchronize()
    ar_ms = sum(a.elapsed_time(b) for a, b in events) / steps
    q.put((rank, sps, ar_ms, len(events) / steps))
    dist.barrier()
    dist.destroy_process_group()


def world2(steps, warmup):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_rank, args=(r, 2, port, steps, warmup, q)) for r in range(2)]
    for p in ps:
        p.start()
    res = sorted(q.get(timeout=1200) for _ in range(2))
    for p in ps:
        p.join(120)
    return res


def old_composition(y, stats, a_out, da, act, gamma):
    """the BatchNorm backward the split kernels replaced"""
    N, H, W, Cn = y.shape
    g = ops.act_bwd(a_out, da, act)
    dx, _ = ops.instnorm_bwd(y, stats, g, ops.ACT_NONE, return_scratch=True)
    unit = torch.zeros((1, Cn, 2), device=y.device, dtype=torch.float64)
    unit[0, :, 1] = H * W * (1.0 - 1e-5)
    return ops.instnorm_apply(dx, unit, ops.ACT_NONE, gammas=gamma.view(1, Cn), betas=torch.zeros((1, Cn), device=y.device),
                              w=torch.ones(1, device=y.device))


def fused(y, stats, da, act, gamma, beta):
    return ops.instnorm_bwd_apply(y, stats, da, ops.instnorm_bwd_reduce(y, stats, da, act, gamma, beta), act, gamma, beta)


def layer_times(reps):
    dev = torch.device("cuda")
    shapes = [("encoder.3", 64, 128, ops.ACT_LRELU), ("encoder.6", 32, 256, ops.ACT_LRELU), ("encoder.9", 16, 512, ops.ACT_LRELU),
              ("decoder.1", 32, 256, ops.ACT_RELU), ("decoder.4", 64, 128, ops.ACT_RELU), ("decoder.7", 128, 64, ops.ACT_RELU)]
    out = []
    for name, hw, c, act in shapes:
        g = torch.Generator(device=dev).manual_seed(hw + c)
        y = torch.randn(1, PER_GPU * hw, hw, c, device=dev, generator=g).bfloat16()
        da = (torch.randn(1, PER_GPU * hw, hw, c, device=dev, generator=g) * 1e-3).bfloat16()
        gamma, beta = torch.rand(c, device=dev, generator=g) + 0.5, torch.randn(c, device=dev, generator=g) * 0.1
        stats = ops.instnorm_stats(y)
        a_out = ops.instnorm_apply(y, stats, act, gammas=gamma.view(1, c), betas=beta.view(1, c), w=torch.ones(1, device=dev))
        runs = {"old": lambda: old_composition(y, stats, a_out, da, act, gamma), "fused": lambda: fused(y, stats, da, act, gamma, beta)}
        for f in runs.values():
            for _ in range(3):
                f()
        t = {k: [] for k in runs}
        for _ in range(5):                   # alternate the two, five rounds of `reps` launches each
            for k, f in runs.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    f()
                e1.record()
                torch.cuda.synchronize()
                t[k].append(e0.elapsed_time(e1) / reps * 1e3)
        old_us, new_us = min(t["old"]), min(t["fused"])
        out.append({"layer": name, "shape": [PER_GPU, hw, hw, c], "MB_bf16": round(y.numel() * 2 / 1e6, 1),
                    "old_us": round(old_us, 1), "fused_us": round(new_us, 1), "speedup": round(old_us / new_us, 2)})
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=50)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("pretrain_dp_bench: needs a CUDA device")
    res = {"card": card(), "gpus": torch.cuda.device_count(), "config": f"Generator({C}) bf16 {RES}x{RES}, {PER_GPU} images/GPU"}
    G, opt = model(torch.device("cuda", 0))
    res["world1_steps_per_s"] = round(steps_per_s(G, opt, data(torch.device("cuda", 0), 100), a.steps, a.warmup), 3)
    del G, opt
    if torch.cuda.device_count() >= 2:
        r = world2(a.steps, a.warmup)
        res["world2_steps_per_s"] = [round(x[1], 3) for x in r]
        res["world2_stat_allreduce_ms_per_step"] = [round(x[2], 3) for x in r]
        res["world2_stat_allreduces_per_step"] = r[0][3]
    else:
        res["world2"] = "not measured: one GPU"
    res["bn_backward_per_layer"] = layer_times(a.reps)
    print(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
