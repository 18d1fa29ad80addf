"""world_size-2 tests (gloo, CPU) of the synchronised-BatchNorm statistics of pretrain.Generator: `bn_batch_stats`, fed
each rank's per-image (sum x, sum x^2), returns the global sums normalised to the rank's own element count and moves the
running statistics exactly as torch.nn.BatchNorm2d(momentum=0.1) in train mode does on the concatenated batch, for even
and uneven shards.  With no group it is the single-process BatchNorm."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

C, HW = 5, (6, 4)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _batch():
    g = torch.Generator().manual_seed(3)
    return torch.randn(4, C, *HW, generator=g, dtype=torch.float64) * 1.7 + 0.4


def _per_image_sums(x):
    """[N, C, 2] = (sum x, sum x^2) per image and channel, as the conv epilogue writes them."""
    return torch.stack([x.sum((2, 3)), (x * x).sum((2, 3))], -1)


def _buffers():
    return torch.zeros(C), torch.ones(C), torch.zeros((), dtype=torch.long)


def _worker(rank, world, port, q, splits):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from multi_style_transfer_gan_b200.pretrain import bn_batch_stats
    x = _batch()
    out = []
    for split in splits:
        lo = sum(split[:rank])
        xs = x[lo:lo + split[rank]]
        M = xs.shape[0] * HW[0] * HW[1]
        rm, rv, nbt = _buffers()
        steps = []
        for _ in range(2):                                   # two updates: the momentum applies to the previous estimate
            stb, scale = bn_batch_stats(_per_image_sums(xs), M, rm, rv, nbt, dist.group.WORLD)
            steps.append((stb.clone(), float(scale)))
        out.append((split, M, steps, rm.clone(), rv.clone(), int(nbt)))
    q.put((rank, out))
    dist.destroy_process_group()


def _reference(x):
    bn = torch.nn.BatchNorm2d(C, momentum=0.1).double().train()
    for _ in range(2):
        bn(x)
    return bn.running_mean, bn.running_var, int(bn.num_batches_tracked)


def test_bn_batch_stats_world2_even_and_uneven_shards():
    world, port = 2, _free_port()
    splits = [(2, 2), (3, 1)]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, world, port, q, splits)) for r in range(world)]
    for p in ps:
        p.start()
    res = dict(q.get(timeout=120) for _ in range(world))
    for p in ps:
        p.join(60)
        assert p.exitcode == 0
    x = _batch()
    glob = _per_image_sums(x).sum(0, keepdim=True)
    M_global = x.shape[0] * HW[0] * HW[1]
    rm_ref, rv_ref, nbt_ref = _reference(x)
    for i, split in enumerate(splits):
        for rank in range(world):
            _, M, steps, rm, rv, nbt = res[rank][i]
            assert M == split[rank] * HW[0] * HW[1]
            for stb, scale in steps:
                assert scale == M / M_global
                # the kernels divide by the LOCAL count: global sums * M / M_global gives the global mean and E[x^2]
                assert torch.allclose(stb, glob * (M / M_global), rtol=1e-14, atol=0), (split, rank)
                assert torch.allclose(stb / M, glob / M_global, rtol=1e-14, atol=0)
            assert torch.allclose(rm.double(), rm_ref, rtol=1e-6, atol=1e-7), (split, rank, rm, rm_ref)
            assert torch.allclose(rv.double(), rv_ref, rtol=1e-6, atol=1e-7), (split, rank, rv, rv_ref)
            assert nbt == nbt_ref
        # every rank holds the same running statistics
        assert torch.equal(res[0][i][3], res[1][i][3]) and torch.equal(res[0][i][4], res[1][i][4])


def test_bn_batch_stats_without_group_is_the_local_batchnorm():
    from multi_style_transfer_gan_b200.pretrain import bn_batch_stats
    x = _batch()[:3]
    M = x.shape[0] * HW[0] * HW[1]
    rm, rv, nbt = _buffers()
    st = _per_image_sums(x)
    for _ in range(2):
        stb, scale = bn_batch_stats(st, M, rm, rv, nbt)
    assert scale is None
    assert torch.equal(stb, st.sum(0, keepdim=True))
    rm_ref, rv_ref, nbt_ref = _reference(x)
    assert torch.allclose(rm.double(), rm_ref, rtol=1e-6, atol=1e-7)
    assert torch.allclose(rv.double(), rv_ref, rtol=1e-6, atol=1e-7)
    assert int(nbt) == nbt_ref


def test_sync_groups_need_an_initialised_world():
    from multi_style_transfer_gan_b200.pretrain import Generator, bn_sync_groups
    G = torch.nn.SyncBatchNorm.convert_sync_batchnorm(Generator(8))
    assert not dist.is_initialized()
    assert bn_sync_groups(G) == {}
