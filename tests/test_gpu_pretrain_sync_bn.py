"""pretrain.Generator trained data-parallel with synchronised BatchNorm (torch.nn.SyncBatchNorm.convert_sync_batchnorm +
DistributedDataParallel): a step on N ranks holding B/N images each equals a single-process step on the B concatenated
images, in outputs, running statistics and gradients, up to the order of floating-point sums.

1. the split BatchNorm backward (msg_instnorm_bwd_reduce / _apply with the affine) against the composition it replaces
   (act_bwd -> instnorm_bwd -> a second apply that multiplies by gamma);
2. a converted model with no process group, or a WORLD of one rank, gives the unconverted model's outputs, input gradient
   and running statistics bit for bit, its parameter gradients up to the fp32 atomics of the weight-gradient kernels, and
   issues no all-reduce;
3. two ranks on ONE GPU over gloo (runs on a single-GPU machine): DDP gradients, running statistics, outputs, three
   pretrain_steps with torch Adam and FusedAdam, and an uneven 3 + 1 split;
4. a training forward + backward issues exactly 12 statistics all-reduces (6 BatchNorm layers x forward / backward),
   an eval forward none;
5. the same over NCCL on two GPUs (skipped with fewer)."""
import io
import os
import socket

import pytest
import torch
import torch.distributed as dist

from tests.util import parity_errors

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


# ---- 1. the split backward kernel -------------------------------------------------------------------------------------
def _bn_views():
    """(H-rows of the [1, N*H, W, C] view, W, C, activation): the six BatchNorm layers of Generator(8) at 64 x 64 with two
    images (encoder: LeakyReLU, decoder: ReLU), and [1, M, 1, 12] planes (C = 12: both dtypes take the generic path)."""
    from multi_style_transfer_gan_b200.ops import ACT_LRELU, ACT_RELU
    gen = [(2 * 16, 16, 16, ACT_LRELU), (2 * 8, 8, 32, ACT_LRELU), (2 * 4, 4, 64, ACT_LRELU),
           (2 * 8, 8, 32, ACT_RELU), (2 * 16, 16, 16, ACT_RELU), (2 * 32, 32, 8, ACT_RELU)]
    syn = [(m, 1, 12, act) for m in (1000, 4099) for act in (ACT_LRELU, ACT_RELU)]
    return gen + syn


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("shape", _bn_views())
def test_split_bn_backward_matches_the_old_composition(shape, dtype):
    from multi_style_transfer_gan_b200 import ops
    from multi_style_transfer_gan_b200.ops import ACT_NONE
    rows, W, C, act = shape
    g = torch.Generator(device=DEV).manual_seed(rows * 131 + C)
    y = (torch.randn(1, rows, W, C, device=DEV, generator=g) * 1.3 + 0.3).to(dtype)
    da = torch.randn(1, rows, W, C, device=DEV, generator=g).to(dtype)
    gamma = torch.randn(C, device=DEV, generator=g) * 0.6 + 0.8
    beta = torch.randn(C, device=DEV, generator=g) * 0.3
    one = torch.ones(1, device=DEV)
    stats = ops.instnorm_stats(y)
    a_out = ops.instnorm_apply(y, stats, act, gammas=gamma.view(1, C), betas=beta.view(1, C), w=one)
    # the composition the split kernels replace
    gin = ops.act_bwd(a_out, da, act)
    dx0, scratch = ops.instnorm_bwd(y, stats, gin, ACT_NONE, return_scratch=True)
    unit = torch.zeros((1, C, 2), device=DEV, dtype=torch.float64)
    unit[0, :, 1] = rows * W * (1.0 - 1e-5)                  # mean 0, var + eps = 1: the apply is dx * gamma
    dx_old = ops.instnorm_apply(dx0, unit, ACT_NONE, gammas=gamma.view(1, C), betas=torch.zeros((1, C), device=DEV), w=one)
    sums = ops.instnorm_bwd_reduce(y, stats, da, act, gamma, beta)
    dx = ops.instnorm_bwd_apply(y, stats, da, sums, act, gamma, beta)
    e_dx, l2_dx = parity_errors(dx.float(), dx_old.float())
    e_db, l2_db = parity_errors(sums[0, :, 0], scratch[0, :, 0])
    e_dg, l2_dg = parity_errors(sums[0, :, 1], scratch[0, :, 1])
    print(f"split bwd {tuple(y.shape)} act {act} {dtype}: dx max {e_dx:.2e} l2 {l2_dx:.2e}; dbeta max {e_db:.2e}; dgamma max {e_dg:.2e}")
    if dtype == torch.float32:
        assert e_dx <= 1e-5, e_dx
        assert e_db <= 1e-6 and e_dg <= 1e-6, (e_db, e_dg)
    else:                                                     # the split path rounds dx once, the composition three times
        assert l2_dx <= 4e-3, l2_dx
        assert l2_db <= 4e-3 and l2_dg <= 4e-3, (l2_db, l2_dg)
    # without the affine the two halves are msg_instnorm_bwd, bit for bit
    plain = ops.instnorm_bwd_apply(y, stats, da, ops.instnorm_bwd_reduce(y, stats, da, act), act)
    assert torch.equal(plain, ops.instnorm_bwd(y, stats, da, act))


# ---- shared model / data -----------------------------------------------------------------------------------------------
def _init_state():
    from multi_style_transfer_gan_b200.pretrain import Generator
    torch.manual_seed(0)
    return {k: v.clone() for k, v in Generator(8).state_dict().items()}


def _data(n=4):
    g = torch.Generator().manual_seed(21)
    real = torch.rand(n, 3, 64, 64, generator=g) * 2 - 1
    mask = (torch.rand(n, 1, 64, 64, generator=g) > 0.4).float().expand(n, 3, 64, 64).contiguous()
    return real * mask, real, mask


def _make(init, dev, sync, precision="fp32"):
    from multi_style_transfer_gan_b200.pretrain import Generator
    G = Generator(8)
    G.load_state_dict(init)
    if sync:
        G = torch.nn.SyncBatchNorm.convert_sync_batchnorm(G)
    return G.to(dev).set_precision(precision).train()


def _running(G):
    return {k: v.detach().cpu().clone() for k, v in G.state_dict().items() if "running" in k or "num_batches" in k}


def _fwd_bwd(G, masked, real, mask, loss="mean"):
    from multi_style_transfer_gan_b200.losses import l1
    x = masked.clone().requires_grad_(True)
    y = G(x)
    inv = 1 - mask
    L = l1(y * inv, real * inv) if loss == "mean" else ((y - real) * inv).abs().sum()
    L.backward()
    return y.detach().cpu(), x.grad.cpu(), float(L.detach())


def _grads(G):
    return {k: p.grad.detach().cpu().clone() for k, p in G.named_parameters()}


class _Counter:
    def __init__(self, fn):
        self.fn, self.n = fn, 0

    def __call__(self, *a, **k):
        self.n += 1
        return self.fn(*a, **k)


# ---- 2. world of one ---------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def test_world_of_one_is_the_unconverted_model(monkeypatch):
    """Outputs, input gradient and running statistics are bit-identical.  Parameter gradients are compared against the
    run-to-run spread of the unconverted model itself: the weight-gradient kernels accumulate with fp32 atomics, so two
    runs of the same model need not agree in the last bits."""
    init = _init_state()
    masked, real, mask = (t.to(DEV) for t in _data())
    ref = _make(init, DEV, sync=False)
    y_ref, dx_ref, _ = _fwd_bwd(ref, masked, real, mask)
    g_ref, run_ref = _grads(ref), _running(ref)
    again = _make(init, DEV, sync=False)
    _fwd_bwd(again, masked, real, mask)
    spread = max(parity_errors(g, g_ref[k])[1] for k, g in _grads(again).items() if not _is_bn_fed_bias(k))
    print(f"unconverted model, two runs: largest parameter-gradient rel-L2 {spread:.2e}")
    counter = _Counter(dist.all_reduce)
    monkeypatch.setattr(dist, "all_reduce", counter)

    def check(G, what):
        y, dx, _ = _fwd_bwd(G, masked, real, mask)
        assert torch.equal(y, y_ref) and torch.equal(dx, dx_ref), what
        run = _running(G)
        assert all(torch.equal(run[k], run_ref[k]) for k in run_ref), what
        for k, g in _grads(G).items():
            if _is_bn_fed_bias(k):
                assert float(g.abs().max()) < 1e-5, (what, k)
            else:
                _close(g, g_ref[k], 2e-6, f"{what} grad {k}", 1e-5)      # two unconverted runs: up to 3.5e-7 on a B200
        assert counter.n == 0, what

    assert not dist.is_initialized()
    check(_make(init, DEV, sync=True), "no process group")
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{_free_port()}", rank=0, world_size=1)
    try:
        check(_make(init, DEV, sync=True), "WORLD of one rank")
    finally:
        dist.destroy_process_group()


# ---- 3 / 4 / 5. two ranks ----------------------------------------------------------------------------------------------
def _worker(rank, world, port, q, backend, init, masked, real, mask):
    import faulthandler
    faulthandler.dump_traceback_later(400, exit=True)       # a hung rank prints its stacks and dies instead of eating the box's time
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dev = torch.device("cuda", rank if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    else:
        dist.init_process_group("gloo", rank=rank, world_size=world)
    from torch.nn.parallel import DistributedDataParallel as DDP

    from multi_style_transfer_gan_b200.enhanced_train import FusedAdam
    from multi_style_transfer_gan_b200.pretrain import pretrain_step
    out = {}

    def shard(split):
        lo = sum(split[:rank])
        return tuple(t[lo:lo + split[rank]].to(dev) for t in (masked, real, mask))

    # 3a. DDP gradients of the local mean loss (averaged by DDP = the global-mean loss), 2 + 2
    m, r, k = shard((2, 2))
    G = _make(init, dev, sync=True)
    D = DDP(G, device_ids=[dev.index])
    y, _, _ = _fwd_bwd(D, m, r, k)
    out["ddp"] = (y, _grads(G), _running(G))
    # 3b. three pretrain_steps: the replicas stay bit-identical (FusedAdam's flat-buffer views survive DDP)
    for name in ("adam", "fused"):
        G = _make(init, dev, sync=True)
        opt = (torch.optim.Adam if name == "adam" else FusedAdam)(G.parameters(), lr=2e-4, betas=(0.5, 0.999))
        D = DDP(G, device_ids=[dev.index])
        losses = [pretrain_step(D, opt, m, r, k) for _ in range(3)]
        views = name == "adam" or all(p.grad.untyped_storage().data_ptr() == opt.flat_grad.untyped_storage().data_ptr()
                                      for p in G.parameters())
        flat = torch.cat([p.detach().reshape(-1) for p in G.parameters()]).cpu()
        out[name] = (losses, flat, _running(G), views)
    # 3c / 4. uneven 3 + 1 without DDP: per-rank gradients of a SUM loss, and the number of statistics all-reduces
    m, r, k = shard((3, 1))
    G = _make(init, dev, sync=True)
    counter = _Counter(dist.all_reduce)
    dist.all_reduce = counter
    try:
        y, _, _ = _fwd_bwd(G, m, r, k, loss="sum")
        n_train = counter.n
        G.eval()
        with torch.no_grad():
            G(m)
        n_eval = counter.n - n_train
    finally:
        dist.all_reduce = counter.fn
    out["uneven"] = (y, _grads(G), _running(G), n_train, n_eval)
    # 5. bf16 forward of the synchronised model, 2 + 2
    m, r, k = shard((2, 2))
    with torch.no_grad():
        out["bf16"] = _make(init, dev, sync=True, precision="bf16")(m).cpu()
    buf = io.BytesIO()                  # bytes, not shared tensors: a rank may exit before the parent reads its result
    torch.save(out, buf)
    q.put((rank, buf.getvalue()))
    dist.barrier()
    dist.destroy_process_group()
    faulthandler.cancel_dump_traceback_later()


def _close(a, b, l2_bound, name, max_bound=None):
    e, l2 = parity_errors(a, b)
    print(f"{name}: max {e:.2e} rel-L2 {l2:.2e}")
    assert l2 <= l2_bound, (name, l2)
    if max_bound is not None:
        assert e <= max_bound, (name, e)


def _is_bn_fed_bias(k):
    """conv biases in front of a BatchNorm: their gradient is analytically zero (the norm removes any per-channel shift)"""
    return k.endswith(".bias") and k.rsplit(".", 1)[0] in ("encoder.2", "encoder.5", "encoder.8", "decoder.0", "decoder.3",
                                                             "decoder.6")


def _run_two_ranks(backend):
    import torch.multiprocessing as mp
    from multi_style_transfer_gan_b200.enhanced_train import FusedAdam  # noqa: F401  (import check before spawning)
    from multi_style_transfer_gan_b200.pretrain import pretrain_step
    init = _init_state()
    masked, real, mask = _data()
    md, rd, kd = (t.to(DEV) for t in (masked, real, mask))
    # single process, the whole batch of four
    ref = _make(init, DEV, sync=False)
    y_ref, _, _ = _fwd_bwd(ref, md, rd, kd)
    g_ref, run_ref = _grads(ref), _running(ref)
    ref = _make(init, DEV, sync=False)
    _fwd_bwd(ref, md, rd, kd, loss="sum")
    g_sum_ref = _grads(ref)
    ref = _make(init, DEV, sync=False)
    loss1_ref = pretrain_step(ref, torch.optim.Adam(ref.parameters(), lr=2e-4, betas=(0.5, 0.999)), md, rd, kd)

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, q, backend, init, masked, real, mask)) for r in range(2)]
    for p in ps:
        p.start()
    res = {r: torch.load(io.BytesIO(b), weights_only=False) for r, b in (q.get(timeout=600) for _ in range(2))}
    for p in ps:
        p.join(120)
        assert p.exitcode == 0
    r0, r1 = res[0], res[1]

    # 3a. outputs, running statistics and DDP gradients
    _close(torch.cat([r0["ddp"][0], r1["ddp"][0]]), y_ref, 1e-5, f"{backend} output", 1e-5)
    for rr in (r0, r1):
        for k, v in run_ref.items():
            assert torch.allclose(rr["ddp"][2][k].double(), v.double(), rtol=1e-5, atol=1e-7), k
        for k, g in g_ref.items():
            if _is_bn_fed_bias(k):
                assert float(rr["ddp"][1][k].abs().max()) < 1e-5, k
            else:
                _close(rr["ddp"][1][k], g, 1e-5, f"{backend} DDP grad {k}")
    # 3b. replicas bit-identical after three steps; the mean of the step-1 local losses is the global-batch loss
    for name in ("adam", "fused"):
        (l0, f0, b0, v0), (l1_, f1, b1, v1) = r0[name], r1[name]
        assert v0 and v1, f"{name}: the optimizer's gradient views did not survive DDP"
        assert torch.equal(f0, f1), name
        assert all(torch.equal(b0[k], b1[k]) for k in b0), name
        avg = 0.5 * (l0[0] + l1_[0])
        assert abs(avg - loss1_ref) <= 1e-5 * abs(loss1_ref), (name, avg, loss1_ref)
        assert not torch.equal(f0, torch.cat([init[k].reshape(-1) for k, _ in ref.named_parameters()])), name
    # 3c. uneven 3 + 1: statistics and outputs as one batch; per-rank gradients of a sum loss add up to the global one
    _close(torch.cat([r0["uneven"][0], r1["uneven"][0]]), y_ref, 1e-5, f"{backend} uneven output", 1e-5)
    for rr in (r0, r1):
        for k, v in run_ref.items():
            assert torch.allclose(rr["uneven"][2][k].double(), v.double(), rtol=1e-5, atol=1e-7), k
    for k, g in g_sum_ref.items():
        s = r0["uneven"][1][k] + r1["uneven"][1][k]
        if _is_bn_fed_bias(k):
            assert float(s.abs().max()) < 1e-5 * y_ref.numel(), k
        else:
            _close(s, g, 1e-5, f"{backend} uneven sum-loss grad {k}")
    # 4. six forward + six backward statistics all-reduces in training, none in eval
    for rr in (r0, r1):
        assert rr["uneven"][3] == 12 and rr["uneven"][4] == 0, rr["uneven"][3:]
    # 5. bf16 tracks fp32 (the bound of the single-GPU pretrain bf16 test)
    _close(torch.cat([r0["bf16"], r1["bf16"]]), y_ref, 5e-2, f"{backend} bf16 vs fp32 output")


def test_two_ranks_on_one_gpu_gloo():
    _run_two_ranks("gloo")


def test_two_gpus_nccl():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    _run_two_ranks("nccl")
