"""GPU: the style-conditional EnhancedGenerator (enable_style_affine / style=) on the sm_100a kernels.

1. msg_style_affine's tables, applied per image, reproduce msg_instnorm_apply's blended affine bit for bit (and the per-image
   backward reduction reproduces the batch-shared one).
2. Identity affines with a one-hot mix give the plain model's forward bit for bit (bf16 c = 64 inference, every fused site;
   fp32), and its conv-weight gradients within the plain model's own run-to-run spread.
3. Random affines and per-image mixes against the CPU restatement (tests/style_affine_oracle.py): fp32 forward at the 1e-4 gate,
   bf16 no worse than 1.25x the plain model's error, fp32 gradients of every conv and affine at the 2e-2 gradient gate, with and
   without gradient checkpointing.
4. Batch independence, 5. the launch list (plain + 1), 6. MultiStyleStylizer with style=."""
import copy

import pytest
import torch

from multi_style_transfer_gan_b200 import _lib, ops
from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
from oracle import restate as R
from tests import style_affine_oracle as O
from tests.util import assert_parity, parity_errors

pytestmark = pytest.mark.gpu
DEV = "cuda"
MIX = torch.tensor([[0.2, 0.3, 0.5], [1.0, 0.0, 0.0], [-0.25, 0.75, 0.5]])


def images(B, H, W, seed):
    return (torch.rand(B, 3, H, W, generator=torch.Generator().manual_seed(seed)) * 2 - 1).to(DEV)


def plain_and_conditional(c, seed, S=3, random_affine=False):
    torch.manual_seed(seed)
    G = EnhancedGenerator(c, 0)
    Gc = copy.deepcopy(G).enable_style_affine(S)
    if random_affine:
        Gc.load_state_dict(O.random_affines(Gc.state_dict(), S, seed + 1))
    return G.to(DEV), Gc.to(DEV)


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("C", [64, 12])
def test_tables_reproduce_the_blended_apply(dtype, C):
    g = torch.Generator().manual_seed(C)
    N, S, H, W = 3, 3, 8, 12
    x = (torch.randn(N, H, W, C, generator=g) * 2 + 0.5).to(DEV, dtype)
    res = torch.randn(N, H, W, C, generator=g).to(DEV, dtype)
    st = ops.instnorm_stats(x)
    gammas = (1 + 0.2 * torch.randn(S, C, generator=g)).to(DEV)
    betas = (0.1 * torch.randn(S, C, generator=g)).to(DEV)
    w = torch.tensor([0.2, 0.3, 0.5], device=DEV)
    tg, tb = ops.style_affine(w.expand(N, S).contiguous(), gammas, betas)
    for r in (None, res):
        ref = ops.instnorm_apply(x, st, ops.ACT_RELU, residual=r, gammas=gammas, betas=betas, w=w)
        out = ops.instnorm_apply(x, st, ops.ACT_RELU, residual=r, affine=(tg.view(-1), tb.view(-1), C))
        assert torch.equal(out, ref)
    # the per-image backward with equal rows is the batch-shared [C] backward
    dy = torch.randn(N, H, W, C, generator=g).to(DEV, dtype)
    g1, b1 = tg[0].contiguous(), tb[0].contiguous()
    sums = ops.instnorm_bwd_reduce(x, st, dy, ops.ACT_RELU, gamma=g1, beta=b1)
    dx = ops.instnorm_bwd_apply(x, st, dy, sums, ops.ACT_RELU, gamma=g1, beta=b1)
    Ct = C + 8                      # rows img_stride apart, other columns untouched
    arena = torch.full((N * Ct * 2,), 7.0, device=DEV, dtype=torch.float64)
    tg2 = torch.zeros(N, Ct, device=DEV)
    tb2 = torch.zeros(N, Ct, device=DEV)
    tg2[:, 8:], tb2[:, 8:] = tg, tb
    aff = (tg2.view(-1)[8:], tb2.view(-1)[8:], Ct)
    ops.instnorm_bwd_reduce_affine(x, st, dy, aff, arena[16:])
    dx2 = ops.instnorm_bwd_apply_affine(x, st, dy, arena[16:], aff)
    a = arena.view(N, Ct, 2)
    assert torch.equal(a[:, 8:], sums) and bool((a[:, :8] == 7.0).all())
    assert torch.equal(dx2, dx)


def test_affine_refused_off_the_tma_kernel():
    g = ops.ConvGeom("conv", 64, 64, 1)
    x = torch.randn(1, 8, 8, 64, device=DEV)                     # fp32: never the TMA kernel
    wp = g.pack_fwd(torch.randn(64, 64, 1, 1, device=DEV), torch.float32)
    st = ops.instnorm_stats(x)
    t = torch.ones(64, device=DEV)
    with pytest.raises(_lib.MsgError, match="error -1"):
        g.forward(x, wp, None, in_stats=st, in_act=ops.ACT_RELU, in_affine=(t, t, 0))


def _names(fn):
    names = []
    _lib.prof_hook, old = (lambda n: names.append(n)), _lib.prof_hook
    try:
        l0 = _lib.launches
        y = fn()
        torch.cuda.synchronize()
        return y, names, _lib.launches - l0
    finally:
        _lib.prof_hook = old


def test_identity_affine_forward_is_bit_exact_and_launches_one_more():
    G, Gc = plain_and_conditional(64, 0)
    x = images(2, 64, 64, 1)
    one_hot = torch.tensor([0.0, 1.0, 0.0])
    with torch.no_grad():
        for prec in ("bf16", "fp32"):
            G.set_precision(prec)
            Gc.set_precision(prec)
            y, names, n = _names(lambda: G(x))
            yc, names_c, nc = _names(lambda: Gc(x, style=one_hot.to(DEV)))
            assert torch.equal(yc, y), prec
            assert nc == n + 1, (prec, n, nc)
            assert names_c.count("msg_style_affine") == 1
            if prec == "bf16":       # every fused site took its affine sibling: the same fused launch list
                for fused in ("msg_down_ring", "msg_la_stage_fwd", "msg_out7_ring", "msg_conv2d"):
                    assert fused + "_affine" in names_c, fused
                assert "msg_instnorm_apply" not in names_c
            assert [k.replace("_affine", "") for k in names_c if k != "msg_style_affine"] == names


def _loss(y, seed):
    r = torch.rand(y.shape, generator=torch.Generator().manual_seed(seed)).to(y.device) * 2 - 1
    return (y * r).sum() / y.numel() + ((y - r) ** 2).mean()


def _grads(G, x, **kw):
    G.zero_grad(set_to_none=True)
    _loss(G(x, **kw), 9).backward()
    return {k: p.grad.detach().clone() for k, p in G.named_parameters() if p.grad is not None}


def test_identity_affine_gradients_within_plain_spread():
    G, Gc = plain_and_conditional(16, 2)
    x = images(2, 32, 32, 3)
    g1, g2 = _grads(G, x), _grads(G, x)
    gc = _grads(Gc, x, style=torch.tensor([1.0, 0.0, 0.0]))
    conv = [k for k in g1 if k.endswith(".0.weight") or ".3." in k]
    spread = max(parity_errors(g2[k], g1[k])[1] for k in conv)
    err = max(parity_errors(gc[k], g1[k])[1] for k in conv)
    assert err <= 2 * spread + 1e-6, (err, spread)


def _oracle_sd(G):
    return {k: v.detach().cpu() for k, v in G.state_dict().items()}


def test_parity_fp32_forward_and_bf16_relative_to_plain():
    # fp32, c = 16: the 1e-4 gate
    _, Gc = plain_and_conditional(16, 4, random_affine=True)
    x = images(3, 64, 48, 5)
    with torch.no_grad():
        y = Gc(x, style=MIX.to(DEV))
    ref = O.generator_forward(_oracle_sd(Gc), x.cpu(), MIX)
    assert_parity(y, ref, 1e-4, "fp32 conditional forward")
    # bf16, c = 64 (the fused inference path): no worse than 1.25x the plain model's error at the same geometry
    G, Gc = plain_and_conditional(64, 6, random_affine=True)
    G.set_precision("bf16")
    Gc.set_precision("bf16")
    x = images(3, 64, 64, 7)
    with torch.no_grad():
        y, yc = G(x), Gc(x, style=MIX.to(DEV))
    e_plain = parity_errors(y, R.generator_forward(_oracle_sd(G), x.cpu()))[1]
    e_cond = parity_errors(yc, O.generator_forward(_oracle_sd(Gc), x.cpu(), MIX))[1]
    assert e_cond <= 1.25 * e_plain, (e_cond, e_plain)


@pytest.mark.parametrize("checkpointing", [False, True])
def test_parity_fp32_gradients(checkpointing):
    _, Gc = plain_and_conditional(16, 8, random_affine=True)
    if checkpointing:
        Gc.gradient_checkpointing_enable()
    x = images(3, 32, 32, 9)
    xg = x.clone().requires_grad_(True)
    _loss(Gc(xg, style=MIX.to(DEV)), 10).backward()
    sd = {k: v.clone().requires_grad_(True) for k, v in _oracle_sd(Gc).items()}
    xr = x.cpu().requires_grad_(True)
    _loss(O.generator_forward(sd, xr, MIX), 10).backward()
    assert_parity(xg.grad, xr.grad, 2e-2, "dx")
    gmax = max(float(v.grad.abs().max()) for v in sd.values() if v.grad is not None)
    n_affine = 0
    for k, p in Gc.named_parameters():
        ref = sd[k].grad
        if ref is None:                        # style_encoder: dead with identity blocks
            continue
        if k.endswith(".0.bias") and not k.startswith("output"):
            # a conv bias in front of an InstanceNorm (affine or not) has an exactly zero gradient
            assert p.grad is None or float(p.grad.abs().max()) == 0.0, k
            assert float(ref.abs().max()) < 1e-4 * gmax, k
            continue
        assert_parity(p.grad, ref, 2e-2, k)
        n_affine += p.dim() == 2
    assert n_affine == 50


def test_batch_independence_with_mixed_styles():
    for c, prec in ((64, "bf16"), (8, "fp32")):
        _, Gc = plain_and_conditional(c, 11, random_affine=True)
        Gc.set_precision(prec)
        x = images(3, 64, 64, 12)
        with torch.no_grad():
            yb = Gc(x, style=MIX.to(DEV))
            for i in range(3):
                yi = Gc(x[i:i + 1], style=MIX[i:i + 1].to(DEV))
                assert_parity(yb[i:i + 1], yi, 2e-6, f"{prec} #{i}")


def test_user_blocks_path_with_style():
    # a user block sends the generator through the encoder / decoder functions: same result as the fused call
    _, Gc = plain_and_conditional(16, 13, random_affine=True)
    x = images(2, 32, 32, 14)
    w = MIX[:2].to(DEV)
    xa = x.clone().requires_grad_(True)
    y0 = Gc(xa, style=w)
    _loss(y0, 3).backward()
    g0 = {k: p.grad.clone() for k, p in Gc.named_parameters() if p.grad is not None}

    class Same(torch.nn.Module):
        def forward(self, t, style, orig):
            return t * 1.0
    Gc.transformer_blocks = torch.nn.ModuleList([Same()])
    Gc.zero_grad(set_to_none=True)
    xb = x.clone().requires_grad_(True)
    y1 = Gc(xb, style=w)
    _loss(y1, 3).backward()
    assert_parity(y1, y0, 1e-5, "y")
    for k, g in g0.items():
        if k.endswith(".1.weight") or k.endswith(".1.bias"):
            assert_parity(Gc.get_parameter(k).grad, g, 1e-4, k)


def _stylizer_gens():
    gens = []
    for s in range(2):
        _, Gc = plain_and_conditional(64, 20 + s, random_affine=True)
        gens.append(Gc)
    return gens


def test_stylizer_with_style():
    gens = _stylizer_gens()
    x = images(3, 64, 64, 15)
    w = [0.6, 0.4]
    serial = MultiStyleStylizer(gens, micro_batch=2, style_streams=False, use_graph=False)
    streams = MultiStyleStylizer(gens, micro_batch=2, style_streams=True, use_graph=False)
    graph = MultiStyleStylizer(gens, micro_batch=2, style_streams=True, use_graph=True)
    for mix in (MIX, MIX[0]):
        ref = serial(x, w, style=mix)
        assert torch.equal(streams(x, w, style=mix), ref)
        assert torch.equal(graph(x, w, style=mix), ref)
    # moving the slider replays the same graph with the new mix
    graph.invalidate_graphs()
    a = graph(x[:2], w, style=MIX[0])
    b = graph(x[:2], w, style=MIX[2])
    assert len(graph._graphs) == 1
    assert torch.equal(a, serial(x[:2], w, style=MIX[0])) and torch.equal(b, serial(x[:2], w, style=MIX[2]))
    assert not torch.equal(a, b)
    # weight maps and uint8 output with a style mix
    maps = torch.rand(1, 2, 4, 4, generator=torch.Generator().manual_seed(16))
    for st in (streams, graph):
        assert torch.equal(st(x, weight_maps=maps, style=MIX, out_uint8=True),
                           serial(x, weight_maps=maps, style=MIX, out_uint8=True))
    # argument checks before any device work
    with pytest.raises(ValueError):
        serial(x, w)
    with pytest.raises(ValueError):
        serial(x, w, style=torch.zeros(2, 3))
    plain = MultiStyleStylizer([EnhancedGenerator(8, 0).to(DEV)], use_graph=False)
    with pytest.raises(ValueError):
        plain(x, [1.0], style=[1.0])
