#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's config, on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload ...] [--dump-outputs DIR]

Workload at N=1 (configs[1]): batch stylisation, 64 synthetic 512x512 images per step, c=64 / 3-block
EnhancedGenerator, 3 styles (3 state dicts, seeds 0..2) blended in output space with weights
[0.2, 0.3, 0.5] (advanced_transform.py:206-213) -- i.e. THREE generator forwards per stylised image,
bf16.  A step = one pass over the batch.  `value` = stylised images/s with inputs resident in HBM;
`e2e` = the same through the public API (MultiStyleStylizer) from pinned HOST fp32 images to HOST
uint8 results, copies inside the timed region.  N>1: one process per GPU (torchrun), images sharded by
rank, no collective on the data path.  The headline is the STATED config: a GLOBAL batch of 64 images sharded 64/N per
GPU ("scaling": "strong"); the weak-scaling point (64 images per GPU) is reported under `weak_scaling`.  The same JSON line
embeds `train` (configs[3]: EnhancedCycleGAN.train_step, batch 8 per GPU, NCCL all-reduce time), and at N=1 `gram`
(configs[2]), `highres` (configs[4]), `cpu_baseline` and `parity` (GPU fp32 / bf16 vs the oracle at 512x512, c=64).

--impl reference: the reference's own CPU implementation of the path (its PyTorch modules restated in
oracle/restate.py -- the reference is not part of this repository) on the host cores, on a bounded sample
(1 image x 3 styles per step).

--dump-outputs DIR: after the timed steps, writes what the timed call returned in its last step as DIR/<name>.npy
(float32 images, float64 losses), so that two builds run with the same arguments -- hence the same seeded inputs and
weights -- can be compared output for output.  An output larger than DUMP_MAX_ELEMS is cut to a fixed, seeded sample of its
elements (dump_sample).  With N > 1 every rank writes its own shard as <name>_rank<r>.npy, sampled to DUMP_MAX_ELEMS / N.

--steps K sets the timed steps of every measurement of the run: the headline, the end-to-end pass, its per-launch
breakdown, and the embedded train, gram, highres and cpu_baseline measurements.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "stylised_images_per_sec_512x512_3styles"
UNIT = "images/s"
STYLE_W = [0.2, 0.3, 0.5]
GEN_GFLOP_512 = 198.844      # BASELINE.md section 3: generator forward, c=64, per 512x512 image
CONV_GFLOP_512 = 181.664     # conv + convT part (SURVEY.md 8d); LocalAttention bmm = 17.180
IN_BYTES_512_BF16 = 520e6    # InstanceNorm algorithmic bytes per image (1 read + 1 write)


def synth_images(B, H, W, seed=1234):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, 3, H, W, generator=g) * 2 - 1


DUMP_MAX_ELEMS = 1 << 23           # 32 MB of float32 over all ranks: the dumps of one run stay under 64 MB


def dump_sample(t, max_elems=DUMP_MAX_ELEMS):
    """t as a host float32 array or, beyond max_elems, a fixed sample of it: the elements at max_elems flat indices drawn
    without replacement by a generator seeded with 0, in increasing order (the same indices for the same shape)."""
    t = t.detach().float()
    if t.numel() > max_elems:
        idx = torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:max_elems].sort().values
        t = t.reshape(-1)[idx.to(t.device)]
    return t.cpu().numpy()


def write_outputs(out_dir, arrays, rank=0, world=1):
    """arrays: {name: numpy float32 / float64 array} -> out_dir/<name>.npy (<name>_rank<r>.npy when world > 1).  Every rank
    writes at most this rank's share of 64 MB, so the dump of the whole run stays under 64 MB."""
    import numpy as np
    assert sum(a.nbytes for a in arrays.values()) * world <= 64e6, "output dump over 64 MB over all ranks"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(out_dir, name + (f"_rank{rank}" if world > 1 else "") + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm_gbs": d["hbm_gbs"], "bf16_tflops": d["bf16_tflops"],
                "bf16_tflops_sustained": d.get("bf16_tflops_sustained", d["bf16_tflops"]), "source": "measured"}
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [t.strip() for t in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------------------------
# reference arm / CPU baseline: the oracle restatement of the reference's PyTorch modules on host cores
# --------------------------------------------------------------------------------------------------
def cpu_reference_images_per_sec(steps, warmup, H=512, W=512, c=64, nb=3, x=None, median=False):
    """Times the oracle port (1 image x 3 styles + blend per step, fp32, all host cores).  Returns
    (images/s, s per step, cores, blended fp32 output of the LAST step) -- the output is the parity anchor of bench.py's
    `parity` block (same weights: seeds 0..2, same image)."""
    from oracle import restate as R
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    cores = os.cpu_count()
    torch.set_num_threads(cores)
    sds = []
    for seed in range(3):
        torch.manual_seed(seed)
        sds.append({k: v.detach() for k, v in EnhancedGenerator(c, nb).state_dict().items()})  # init only, CPU
    if x is None:
        x = synth_images(1, H, W)
    times, y = [], None
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            ys = [R.generator_forward(sd, x) for sd in sds]
            y = R.blend_outputs(ys, STYLE_W)
            R.to_uint8_image(y)
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    times.sort()
    per_step = times[len(times) // 2] if median else sum(times) / len(times)
    return 1.0 / per_step, per_step, cores, y


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    v, per_step, cores, y = cpu_reference_images_per_sec(args.steps, args.warmup)
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"stylised": dump_sample(y)})
    line = {"metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": per_step * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "impl": "reference",
            "config": {"workload": "batch stylisation 512x512, c=64/3-block generator, 3 styles blended [0.2,0.3,0.5]",
                       "sample": "1 image x 3 styles per step (of the 64-image batch)",
                       "note": "the reference is 100 % Python (stock torch.nn modules) and not part of this repository, "
                               "so this arm runs its restatement oracle/restate.py (kind 'port'), which is pinned to the "
                               "unmodified reference by tests/golden/ (bit-identical init, <= 1e-4 outputs)"},
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": "1 image x 3 generator forwards + blend per step, fp32, torch CPU (oracle/restate.py)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------------
def csrc_digest():
    """sha256 over the kernel sources: the ncu-measured DRAM traffic in profiles/traffic.json is only quoted for the exact
    sources it was measured on (a stale number is worse than none)."""
    import hashlib
    d = os.path.join(ROOT, "multi_style_transfer_gan_b200", "csrc")
    h = hashlib.sha256()
    for f in sorted(os.listdir(d)):
        with open(os.path.join(d, f), "rb") as fh:
            h.update(f.encode() + b"\0" + fh.read())
    return h.hexdigest()[:16]


def standalone_apply_elems(per_fwd, c, H, W):
    """elements moved per image by the stand-alone IN apply launches of one forward.  8 of the 13 applies are always fused into their
    consumers (no HBM pass).  5 left: the initial IN (1 read + 1 write of [c, H, W]) and the four MultiScaleBlock outputs (read +
    residual read + write).  3 left (c = 64 inference with the fused down / output ring kernels): the MultiScaleBlock outputs of
    down1, down2 and up1."""
    msb3 = 3 * (2 * (2 * c) * (H // 2) * (W // 2) + (4 * c) * (H // 4) * (W // 4))
    if per_fwd == 3:
        return msb3
    return c * H * W * 2 + msb3 + 3 * c * H * W


def measured_traffic(key, micro_batch=None):
    """profiles/traffic.json: {"csrc_sha": ..., "ncu_file": ..., key: bytes per launch}; None when absent or stale."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None, "no ncu capture committed for these sources"
    d = json.load(open(p))
    if d.get("csrc_sha") != csrc_digest():
        return None, f"stale: {d.get('ncu_file')} was captured on csrc {d.get('csrc_sha')}, sources are now {csrc_digest()}"
    if micro_batch is not None and d.get("micro_batch", 16) != micro_batch:
        return None, f"{d.get('ncu_file')} was captured at micro-batch {d.get('micro_batch', 16)}, this run uses {micro_batch}"
    return d.get(key), f"dram__bytes_read.sum + dram__bytes_write.sum per launch, {d.get('ncu_file')} (csrc {d.get('csrc_sha')})"


class Ctx:
    """rank / device / timing helpers shared by the sub-benchmarks of one bench.py process"""

    def __init__(self):
        import torch.distributed as dist
        self.dist = dist
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(self, v):
        if self.world > 1:
            t = torch.tensor([v], device=self.dev, dtype=torch.float64)
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
            return float(t.item())
        return v

    def timed(self, fn, steps, warmup, prof=False):
        """W untimed warm-ups, then exactly K steps between barrier + synchronize, CUDA events, max over ranks."""
        from multi_style_transfer_gan_b200 import _lib, profiler
        for _ in range(warmup):
            fn()
        self.barrier()
        l0 = _lib.launches
        if prof:
            profiler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = e0.elapsed_time(e1)
        breakdown = profiler.stop() if prof else None
        return self.max_over_ranks(ms) / steps, _lib.launches - l0, breakdown


def bench_stylise(cx, args, gens, B_rank, seed_off=0, want_breakdown=True, want_e2e=True, want_output=False):
    """One stylisation measurement with B_rank images on this rank.  Returns a dict of per-step times (max over ranks) and,
    with want_output, the (sampled) images of the last timed step under "output"."""
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    H = W = args.size
    sty = MultiStyleStylizer(gens, precision=args.precision, micro_batch=args.micro_batch)
    x_host = synth_images(B_rank, H, W, seed=1234 + seed_off).pin_memory()
    x_dev = x_host.to(cx.dev)
    out_dev = torch.empty((B_rank, 3, H, W), device=cx.dev, dtype=torch.float32)
    out_host = torch.empty((B_rank, 3, H, W), dtype=torch.uint8).pin_memory()
    # inputs (64 x 512^2 fp32 = 201 MB at N=1; >= 25 MB + the activations of a micro-batch, > 1 GB, at N=8) exceed the
    # 126 MB L2, so nothing is L2-resident between timed iterations (no explicit flush needed).
    r = {"sty": sty, "x_host": x_host, "out_host": out_host}
    r["ms_dev"], r["launches"], _ = cx.timed(lambda: sty(x_dev, STYLE_W, out=out_dev), args.steps, args.warmup)
    if want_output:                        # before the passes below overwrite out_dev
        r["output"] = dump_sample(out_dev, DUMP_MAX_ELEMS // cx.world)
    if want_breakdown:
        # per-launch CUDA-event breakdown (roofline): the same step with one stream and no graph replay, because launches
        # inside a replayed graph cannot be bracketed by events and concurrent kernels of different styles share the SMs
        sty_serial = MultiStyleStylizer(gens, precision=args.precision, micro_batch=args.micro_batch, style_streams=False,
                                        use_graph=False)
        r["ms_serial"], _, r["breakdown"] = cx.timed(lambda: sty_serial(x_dev, STYLE_W, out=out_dev), args.steps, 1, prof=True)
    if want_e2e:
        # the public API with HOST buffers: pinned fp32 in -> uint8 out, both copies inside the timed region (the call
        # returns when the last D2H copy has landed)
        r["ms_e2e"], _, _ = cx.timed(lambda: sty(x_host, STYLE_W, out_uint8=True, out=out_host), args.steps, 1)
    return r


def roofline_blocks(args, B_rank, breakdown, ms_serial, pk):
    """roofline of the dominant kernel family (every tensor-core launch of the step: convs, transposed convs and the fused /
    stand-alone LocalAttention stages) and of the stand-alone InstanceNorm applies, from the serialised pass."""
    H = W = args.size
    scale = (H * W) / 512 ** 2
    out = {}
    conv_keys = ("msg_conv2d", "msg_conv_slab", "msg_conv_shift", "msg_msb64_ring", "msg_msb_ring", "msg_convt_ring", "msg_out7_ring", "msg_down_ring", "msg_la_stage_fwd",
                 "msg_local_attn_fwd")
    conv_ms = sum(breakdown.get(k, {}).get("ms", 0.0) for k in conv_keys) / args.steps
    conv_launches = sum(breakdown.get(k, {}).get("launches", 0) for k in conv_keys) // args.steps
    fused_la = breakdown.get("msg_la_stage_fwd", {}).get("launches", 0) > 0
    # algorithmic flops of those launches: conv + convT + the two LocalAttention contractions (BASELINE.md 3: 198.844 GFLOP per
    # 512x512 forward).  The attention products run inside the fused stage kernel (tcgen05) at C = 64 / 128 and in the
    # stand-alone attention kernel (mma.sync) at C = 256: both are tensor-core launches of this family.
    gflop = GEN_GFLOP_512
    flops = 3 * B_rank * gflop * scale * 1e9
    if conv_ms > 0:
        ach = flops / (conv_ms * 1e-3) / 1e12
        traffic, tnote = (measured_traffic("conv_dram_bytes_per_launch", args.micro_batch) if (H == 512 and args.channels == 64
                                                                              and B_rank % args.micro_batch == 0) else (None, "not the profiled configuration"))
        out["roofline"] = {"bound": "tensor",
                           "kernel": "conv_tma_kernel + conv_slab_kernel + conv_shift_kernel"
                                     + (" + msb_ring_kernel" if (breakdown.get("msg_msb64_ring", {}).get("launches", 0)
                                                                 or breakdown.get("msg_msb_ring", {}).get("launches", 0)) else "")
                                     + (" + convt_ring_kernel" if breakdown.get("msg_convt_ring", {}).get("launches", 0) else "")
                                     + (" + out7_ring_kernel" if breakdown.get("msg_out7_ring", {}).get("launches", 0) else "")
                                     + (" + down_ring_kernel" if breakdown.get("msg_down_ring", {}).get("launches", 0) else "")
                                     + (" + la_stage_kernel" if fused_la else "")
                                     + (" + local_attn_fwd_tc_kernel" if breakdown.get("msg_local_attn_fwd", {}).get("launches", 0) else "")
                                     + " (every tensor-core launch of the step)",
                           "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                           "frac": ach / pk["bf16_tflops_sustained"], "traffic": traffic, "traffic_note": tnote,
                           "algorithmic_gflop_per_image_forward": gflop * scale,
                           "peak_source": pk["source"] + " (sustained bf16; kernel timed inside a long step)",
                           "launches_per_step": conv_launches, "ms_per_step": conv_ms,
                           "launches_note": "C-ABI calls; msg_msb_ring at C = 128 is 3 kernels per call, msg_convt_ring and msg_down_ring 2",
                           "measured_on": f"serialised pass of the same step (one stream, no graph replay, {ms_serial:.1f} ms per step): "
                                          "launches inside a replayed graph cannot be bracketed by events"}
    in_keys = ("msg_instnorm_apply", "msg_instnorm_stats")
    in_ms = sum(breakdown.get(k, {}).get("ms", 0.0) for k in in_keys) / args.steps
    if in_ms > 0:
        in_launches = sum(breakdown.get(k, {}).get("launches", 0) for k in in_keys) // args.steps
        per_fwd = in_launches // (3 * max(1, (B_rank + args.micro_batch - 1) // args.micro_batch))
        c = args.channels
        if per_fwd <= 5:
            in_bytes = standalone_apply_elems(per_fwd, c, H, W) * 2
            note = f"{per_fwd} stand-alone apply launches per forward (the others are fused into their consumers)"
        else:
            in_bytes, note = IN_BYTES_512_BF16 * scale, "13 apply launches per forward, 1 read + 1 write each (SURVEY 8d)"
        gbs = 3 * B_rank * in_bytes / (in_ms * 1e-3) / 1e9
        out["roofline_instnorm"] = {"bound": "hbm", "achieved": gbs, "peak": pk["hbm_gbs"], "unit": "GB/s",
                                    "frac": gbs / pk["hbm_gbs"], "ms_per_step": in_ms, "bytes": note}
    out["breakdown_ms_per_step"] = {k: round(v["ms"] / args.steps, 3) for k, v in sorted(breakdown.items(), key=lambda kv: -kv[1]["ms"])}
    return out


# wgrad GEMM flops of one train step at c=64, 256x256 (BASELINE.md section 3: conv + convT flops of a generator forward =
# 181.664 / 4 GFLOP per image at 256^2, discriminator 4.537): 6 generator backward passes (fake, identity, cycle for each of
# G_AB / G_BA) and 4 discriminator backward passes with weight gradients (the D phase), per image
TRAIN_WGRAD_GFLOP_PER_IMAGE = 6 * (CONV_GFLOP_512 / 4) + 4 * 4.537


def bench_train(cx, args, steps, warmup):
    """BASELINE.json configs[3]: EnhancedCycleGAN.train_step, c=64, batch 8 per GPU at 256x256, bf16, data-parallel with one
    flat NCCL all-reduce per optimizer per step (weak scaling: 8 images per GPU)."""
    from multi_style_transfer_gan_b200 import _lib, profiler
    from multi_style_transfer_gan_b200.enhanced_train import EnhancedCycleGAN
    torch.manual_seed(0)
    c = args.channels
    style = None
    if args.lambda_style > 0:                  # + VGG-19 Gram style term (random-init trunk, seed 0)
        from multi_style_transfer_gan_b200.style_loss import GramStyleLoss, VGG19Features
        style = GramStyleLoss(VGG19Features(cx.dev, seed=0), precision=args.precision)
    use_graph = not args.no_train_graph
    m = EnhancedCycleGAN(channels=c, num_transformer_blocks=3 if c == 64 else 1, precision=args.precision, device=cx.dev,
                         style_loss=style, lambda_style=args.lambda_style, use_graph=use_graph, graph_warmup=2)
    B, S = args.train_batch, args.train_size
    A = synth_images(B, S, S, seed=11 + cx.rank).pin_memory()
    Bm = synth_images(B, S, S, seed=12 + cx.rank).pin_memory()
    n_eager = 2
    for _ in range(n_eager):
        m.train_step(A, Bm)
    torch.cuda.synchronize()
    # the collectives on their own: the two flat-gradient all-reduces of a step (discriminators, generators), CUDA events on the
    # launching stream, after two untimed rounds.  In the step the first one runs under the identity forwards.
    comm_ms, comm_bytes, comm_calls = 0.0, 0, 0
    if cx.world > 1:
        bufs = [m.d_optimizer.flat_grad, m.g_optimizer.flat_grad]
        for _ in range(2):
            for b_ in bufs:
                cx.dist.all_reduce(b_)
        cx.barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        for _ in range(5):
            for b_ in bufs:
                cx.dist.all_reduce(b_)
        c1.record()
        torch.cuda.synchronize()
        comm_ms = cx.max_over_ranks(c0.elapsed_time(c1) / 5)
        comm_bytes, comm_calls = sum(b_.numel() * 4 for b_ in bufs), len(bufs)
        for b_ in bufs:
            b_.zero_()
    for _ in range(max(0, warmup - n_eager) + (1 if use_graph else 0)):      # (+ the capturing step)
        m.train_step(A, Bm)
    cx.barrier()
    l0 = _lib.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        losses = m.train_step(A, Bm)       # host fp32 batches in (pinned), five loss floats out: the public API, H2D/D2H inside
    e1.record()
    cx.barrier()
    ms = cx.max_over_ranks(e0.elapsed_time(e1) / steps)
    launches_per_step = (_lib.launches - l0) // steps
    graphed = m._graph is not None
    # per-entry-point breakdown: one more step run eagerly (same kernels; a replayed graph cannot be bracketed by events)
    m.use_graph = False
    profiler.start()
    m.train_step(A, Bm)
    breakdown = profiler.stop()
    bsteps = 1
    pk = peaks()
    wg_ms = breakdown.get("msg_conv2d_wgrad", {}).get("ms", 0.0) / bsteps
    out = {"metric": "train_steps_per_sec", "value": 1e3 / ms, "unit": "steps/s", "ms_per_step": ms, "steps": steps, "warmup": warmup,
           "scaling": "weak", "dtype": "bf16" if args.precision == "bf16" else "f32",
           "config": {"workload": "EnhancedCycleGAN.train_step (2 G + 2 D, LSGAN + cycle + identity + structure losses"
                                  + (f" + {args.lambda_style:g} x VGG-19 Gram style loss (random-init trunk)" if style else "")
                                  + f", fused Adam), c={c}, batch {B} per GPU at {S}x{S}",
                      "global_batch": B * cx.world, "parallelism": f"data-parallel x{cx.world}, 2 flat NCCL all-reduces per step",
                      "schedule": (f"step replayed as {len(m._graph['graphs'])} CUDA-graph segment(s)"
                                   + (", the NCCL all-reduces eager between them" if len(m._graph["graphs"]) > 1 else "")) if graphed else
                                  ("eager launches" + (f" (graph capture failed: {m.graph_error})" if m.graph_error else ""))},
           "images_per_sec": B * cx.world * 1e3 / ms,
           "gpu_launches_per_step": launches_per_step, "losses": losses,
           "nccl": {"ms_per_step": comm_ms, "bytes_per_step": comm_bytes, "calls_per_step": comm_calls,
                    "how": "the step's two flat-gradient all-reduces timed on their own (CUDA events on the launching stream, 5 rounds "
                           "after 2 warm-up rounds, max over ranks); in the step the discriminator one runs under the identity forwards"},
           "e2e": {"value": 1e3 / ms, "unit": "steps/s", "h2d_bytes_per_step": 2 * A.numel() * 4, "d2h_bytes_per_step": 20},
           "breakdown_ms_per_step": {k: round(v["ms"] / bsteps, 3) for k, v in sorted(breakdown.items(), key=lambda kv: -kv[1]["ms"])[:12]},
           "breakdown_note": "one eager step after the timed region (same kernels)"}
    if wg_ms > 0 and c == 64 and S == 256:
        ach = TRAIN_WGRAD_GFLOP_PER_IMAGE * B * 1e9 / (wg_ms * 1e-3) / 1e12
        out["roofline_wgrad"] = {"bound": "tensor", "kernel": "conv_wgrad_tc_kernel (every weight-gradient launch of the step)",
                                 "achieved": ach, "peak": pk["bf16_tflops_sustained"], "unit": "TFLOP/s",
                                 "frac": ach / pk["bf16_tflops_sustained"], "ms_per_step": wg_ms,
                                 "launches_per_step": breakdown["msg_conv2d_wgrad"]["launches"] // bsteps}
    del m
    torch.cuda.empty_cache()
    return out


def bench_gram(cx, args):
    """BASELINE.json configs[2]: Gram-matrix style loss forward + backward on the five VGG-19 tap shapes, batch 16 at 256x256
    (kernel-only, bf16 features = relu(randn)), and the same with the VGG-19 trunk forward + backward to the image."""
    from multi_style_transfer_gan_b200 import ops
    from multi_style_transfer_gan_b200.style_loss import GramStyleLoss, VGG19Features
    dev = cx.dev
    torch.manual_seed(0)
    shapes = [(64, 256), (128, 128), (256, 64), (512, 32), (512, 16)]
    feats = [torch.relu(torch.randn(16, s, s, c, device=dev)).to(torch.bfloat16) for c, s in shapes]
    tgts = [ops.gram(f) for f in feats]

    def gram_fb():
        loss = torch.zeros(1, device=dev)
        for f, t in zip(feats, tgts):
            _, g = ops.gram_loss_fwd(f, t, 1.0, loss)
            ops.gram_loss_bwd(f, g, t, 1.0)

    ms, _, _ = cx.timed(gram_fb, args.steps, 3)
    fl = 2 * sum(2.0 * c * c * s * s * 16 for c, s in shapes)            # fwd + bwd, 2*C^2*HW each
    by = sum(f.numel() * 2 * 3 for f in feats)                           # features read twice (fwd, bwd) + dF written
    pk = peaks()
    vgg = VGG19Features(dev, seed=0)
    sl = GramStyleLoss(vgg, "bf16").set_style(torch.rand(16, 3, 256, 256, device=dev) * 2 - 1)
    y = (torch.rand(16, 3, 256, 256, device=dev) * 2 - 1).requires_grad_(True)

    def full():
        y.grad = None
        sl(y).backward()

    ms_full, _, _ = cx.timed(full, args.steps, 3)
    return {"config": "Gram + style-loss forward + backward, VGG-19 relu1_1..relu5_1 shapes, batch 16 at 256x256, bf16",
            "ms": ms, "tflops_algorithmic": fl / ms / 1e9, "feature_gbs": by / ms / 1e6,
            "hbm_frac": by / ms / 1e6 / pk["hbm_gbs"], "parity": "unpinned (not in the reference; trunk pinned to torchvision, "
            "tests/test_oracle_vgg_torchvision.py)",
            "with_vgg19_trunk": {"ms": ms_full, "images_per_sec": 16e3 / ms_full,
                                 "what": "VGG-19 features[:30] forward, Gram loss, backward to the image (random-init trunk)"}}


def bench_highres(cx, args):
    """BASELINE.json configs[4]: 1024x1024, batch 8, 4 blended styles, c=64: throughput, peak memory, IN bandwidth."""
    from multi_style_transfer_gan_b200 import profiler
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    gens = []
    for s in range(4):
        torch.manual_seed(s)
        gens.append(EnhancedGenerator(64, 3).to(cx.dev))
    w4 = [0.4, 0.3, 0.2, 0.1]
    st = MultiStyleStylizer(gens, precision=args.precision, micro_batch=4)
    x = synth_images(8, 1024, 1024, seed=5).to(cx.dev)
    torch.cuda.reset_peak_memory_stats()
    ms, _, _ = cx.timed(lambda: st(x, w4), args.steps, 2)
    peak_gib = torch.cuda.max_memory_allocated() / 2 ** 30
    ser = MultiStyleStylizer(gens, precision=args.precision, micro_batch=4, style_streams=False, use_graph=False)
    _, _, bd = cx.timed(lambda: ser(x, w4), args.steps, 1, prof=True)
    pk = peaks()
    out = {"config": "1024x1024, batch 8, 4 styles blended [0.4,0.3,0.2,0.1], c=64/3-block, bf16, micro-batch 4",
           "ms_per_batch": ms, "images_per_sec": 8e3 / ms, "peak_memory_gib": peak_gib}
    in_ms = bd.get("msg_instnorm_apply", {}).get("ms", 0.0) / args.steps
    n = bd.get("msg_instnorm_apply", {}).get("launches", 0) // args.steps
    if in_ms > 0:
        per_fwd = n // (4 * 2)
        H = W = 1024
        c = 64
        elems = standalone_apply_elems(per_fwd, c, H, W) if per_fwd <= 5 else IN_BYTES_512_BF16 * 4 / 2
        gbs = 4 * 8 * elems * 2 / (in_ms * 1e-3) / 1e9
        out["instnorm"] = {"gbs": gbs, "hbm_frac": gbs / pk["hbm_gbs"], "ms": in_ms, "standalone_apply_launches_per_forward": per_fwd}
    del gens, st, ser
    torch.cuda.empty_cache()
    return out


def bench_parity(cx, args, gens, x0, y_oracle):
    """Parity at the benchmark geometry: image 0 x 3 styles at 512x512, c=64, against the oracle's blended fp32 output (computed
    in the cpu_baseline leg).  fp32 engine: the <= 1e-4 gate of BASELINE.md section 4; bf16 hot path: max-abs and rel-L2 reported."""
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    out = {"what": f"image 0 of the batch x 3 styles, {args.size}x{args.size}, c={args.channels}, vs oracle/restate.py fp32 (CPU)"}
    ref = y_oracle.to(cx.dev)
    for prec in ("fp32",) + (("bf16",) if args.precision == "bf16" else ()):
        sty = MultiStyleStylizer(gens, precision=prec, micro_batch=1, style_streams=False, use_graph=False)
        y = sty(x0.to(cx.dev), STYLE_W)
        torch.cuda.synchronize()
        d = (y - ref).float()
        out[prec] = {"max_abs": float(d.abs().max()), "rel_l2": float(d.norm() / ref.norm()),
                     "max_abs_over_max_ref": float(d.abs().max() / ref.abs().max())}
    for g in gens:
        g.set_precision(args.precision)
    out["fp32"]["gate"] = "<= 1e-4 rel-L2 (BASELINE.md 4)"
    out["fp32"]["ok"] = out["fp32"]["rel_l2"] <= 1e-4
    return out


def run_ours(args):
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    from multi_style_transfer_gan_b200.stylize import shard_range
    cx = Ctx()
    rank, world = cx.rank, cx.world
    H = W = args.size
    c, nb = args.channels, 3 if args.channels == 64 else 1
    gens = []
    for seed in range(3):
        torch.manual_seed(seed)
        gens.append(EnhancedGenerator(c, nb).to(cx.dev))
    B = args.batch                        # GLOBAL batch of the headline (BASELINE.json configs[1]: 64 images, sharded 64/N)
    lo, hi = shard_range(B, rank, world)
    sampler = ClockSampler(cx.local)
    if rank == 0:
        sampler.start()
    main = bench_stylise(cx, args, gens, hi - lo, seed_off=rank, want_output=bool(args.dump_outputs))
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"stylised": main.pop("output")}, rank, world)
    weak = None
    if world > 1:                         # the weak-scaling point of round 1 (64 images per GPU), kept as an extra key
        w = bench_stylise(cx, args, gens, B, seed_off=rank, want_breakdown=False, want_e2e=False)
        weak = {"value": world * B / (w["ms_dev"] * 1e-3), "unit": UNIT, "ms_per_step": w["ms_dev"], "batch_per_gpu": B,
                "global_batch": world * B, "scaling": "weak"}
    clocks = sampler.stop() if rank == 0 else None
    ms_dev, ms_e2e = main["ms_dev"], main["ms_e2e"]
    sty = main["sty"]
    pk = peaks()
    line = {"metric": METRIC, "value": B / (ms_dev * 1e-3), "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_dev, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "bf16" if args.precision == "bf16" else "f32", "data": "synthetic",
            "config": {"workload": f"batch stylisation {H}x{W}, GLOBAL batch {B} sharded {hi - lo} images per GPU, 3 style weights {STYLE_W}, "
                                   f"c={c}/{nb}-block EnhancedGenerator, reference-faithful output blend = 3 generator "
                                   f"forwards per image ({3 * GEN_GFLOP_512 * (H * W) / 512 ** 2:.1f} GFLOP/image)",
                       "global_batch": B, "batch_per_gpu": hi - lo, "micro_batch": args.micro_batch,
                       "schedule": f"style_streams={int(sty.style_streams)}, cuda_graph={int(sty.use_graph)}",
                       "parallelism": f"image-sharded x{world}, no collective on the data path",
                       "l2": "inputs + per-micro-batch activations > 126 MB L2; no flush needed",
                       "weights": "random init (seeds 0,1,2), fp32 master, bf16 packed"},
            "gpu_launches": main["launches"],
            "e2e": {"value": B / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": main["x_host"].numel() * 4,
                    "d2h_bytes_per_step": main["out_host"].numel(), "ms_per_step": ms_e2e,
                    "what": "MultiStyleStylizer(host pinned fp32 -> host uint8), per-rank bytes"},
            "clocks": clocks}
    if weak is not None:
        line["weak_scaling"] = weak
    if main.get("breakdown") and rank == 0:
        line.update(roofline_blocks(args, hi - lo, main["breakdown"], main["ms_serial"], pk))
    del main
    torch.cuda.empty_cache()
    if not args.no_extras:
        # BASELINE.json configs[3] (train step, every N: the only data-path collective of the repo), configs[2] and configs[4] (N = 1)
        try:
            t = bench_train(cx, args, steps=args.steps, warmup=3)
            if rank == 0:
                line["train"] = t
        except Exception as e:           # the headline must survive a failure of a secondary workload -- but loudly
            if rank == 0:
                line["train"] = {"error": repr(e)}
        if world == 1:
            for key, fn in (("gram", lambda: bench_gram(cx, args)), ("highres", lambda: bench_highres(cx, args))):
                try:
                    line[key] = fn()
                except Exception as e:
                    line[key] = {"error": repr(e)}
    if rank == 0:
        if world == 1 and not args.no_cpu_baseline:
            x0 = synth_images(B, H, W, seed=1234)[0:1].contiguous()
            v, per_step, cores, y_ref = cpu_reference_images_per_sec(args.steps, 2, H, W, c, nb, x=x0, median=True)
            line["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "1 image x 3 generator forwards + blend, fp32, torch CPU restatement of the "
                                              f"reference modules (oracle/restate.py), 2 warm-ups + median of {args.steps}"}
            try:
                line["parity"] = bench_parity(cx, args, gens, x0, y_ref)
            except Exception as e:
                line["parity"] = {"error": repr(e)}
        print(json.dumps(line))
    if world > 1:
        cx.dist.destroy_process_group()


def run_train(args):
    """Secondary workload on its own (BASELINE.json configs[3]); the default run embeds the same measurement as `train`."""
    cx = Ctx()
    t = bench_train(cx, args, steps=args.steps, warmup=args.warmup)
    if args.dump_outputs:                  # the five losses train_step returned in the last timed step
        import numpy as np
        write_outputs(args.dump_outputs, {f"train_{k}": np.array(v, dtype=np.float64) for k, v in t["losses"].items()},
                      cx.rank, cx.world)
    if cx.rank == 0:
        line = {"n_gpus": cx.world, "higher_is_better": True, "vs_baseline": None, "data": "synthetic"}
        line.update(t)
        print(json.dumps(line))
    if cx.world > 1:
        cx.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of every measurement of the run (see the module docstring)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--channels", type=int, default=64)
    ap.add_argument("--micro-batch", type=int, default=32)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the embedded train / gram / highres measurements")
    ap.add_argument("--workload", default="stylise", choices=["stylise", "train"])
    ap.add_argument("--no-train-graph", action="store_true", help="train workload: eager launches instead of one CUDA-graph replay per step")
    ap.add_argument("--train-batch", type=int, default=8)
    ap.add_argument("--train-size", type=int, default=256)
    ap.add_argument("--lambda-style", type=float, default=0.0,
                    help="train workload: weight of the VGG-19 Gram style term (0 = the reference's train_step)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed call returned in its last step to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.impl == "reference":
        run_reference(args)
    else:
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device (the msg_b200 path has no CPU fallback); use --impl reference for the CPU arm")
        (run_train if args.workload == "train" else run_ours)(args)


if __name__ == "__main__":
    main()
