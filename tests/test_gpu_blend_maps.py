"""GPU: the per-pixel blend (msg_blend_maps) and map feathering (msg_gaussian_blur) against their CPU restatement (tests/blend_maps_oracle.py), their exact
properties (constant maps reproduce msg_blend_outputs bit for bit), and MultiStyleStylizer's weight_maps under every
schedule."""
import pytest
import torch


pytestmark = pytest.mark.gpu
DEV = "cuda"


def rand(*shape, seed=0, lo=-1.0, hi=1.0):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(*shape, generator=g) * (hi - lo) + lo


@pytest.mark.parametrize("hw", ["1x1", "5x7", "quarter", "full"])
@pytest.mark.parametrize("per_image", [False, True])
@pytest.mark.parametrize("with_x", [False, True])
@pytest.mark.parametrize("normalize", [False, True])
@pytest.mark.parametrize("HW", [(24, 40), (20, 37)])          # W % 4 == 0 (vector path) and not (scalar path)
def test_blend_maps_matches_oracle(hw, per_image, with_x, normalize, HW):
    from multi_style_transfer_gan_b200 import ops
    from oracle import restate as R
    from tests import blend_maps_oracle as BM
    N, C, S = 3, 3, 3
    H, W = HW
    h, w = {"1x1": (1, 1), "5x7": (5, 7), "quarter": (H // 4, W // 4), "full": (H, W)}[hw]
    ys = [rand(N, C, H, W, seed=s) for s in range(S)]
    x = rand(N, C, H, W, seed=10)
    K = S + 1 if with_x else S
    maps = rand(N if per_image else 1, K, h, w, seed=20, lo=0.0, hi=1.0)
    out, u8 = ops.blend_maps([y.to(DEV) for y in ys], maps.to(DEV), x=x.to(DEV) if with_x else None, gain=1.1,
                             clip=(-0.9, 0.9), normalize=normalize, out_uint8=True)
    ref = BM.blend_maps(ys, maps, x=x if with_x else None, gain=1.1, clip=(-0.9, 0.9), normalize=normalize)
    assert float((out.cpu() - ref).abs().max()) <= 1e-6
    assert torch.equal(u8.cpu(), R.to_uint8_image(out.cpu()))
    u8_only = torch.empty_like(u8)
    ops.blend_maps([y.to(DEV) for y in ys], maps.to(DEV), x=x.to(DEV) if with_x else None, gain=1.1, clip=(-0.9, 0.9),
                   normalize=normalize, out=u8_only)
    assert torch.equal(u8_only, u8)


@pytest.mark.parametrize("HW", [(16, 24), (15, 21)])
def test_constant_maps_equal_blend_outputs(HW):
    from multi_style_transfer_gan_b200 import ops
    N, C, S = 2, 3, 3
    ys = [rand(N, C, *HW, seed=s).to(DEV) for s in range(S)]
    x = rand(N, C, *HW, seed=9).to(DEV)
    w, w_x = [0.2, 0.3, 0.5], 0.35
    m = torch.tensor(w + [w_x], device=DEV).view(1, S + 1, 1, 1)
    assert torch.equal(ops.blend_maps(ys, m[:, :S].contiguous(), gain=1.1, clip=(-1, 1)),
                       ops.blend_outputs(ys, w, gain=1.1, clip=(-1, 1)))
    f, u = ops.blend_maps(ys, m.contiguous(), x=x, out_uint8=True)
    rf, ru = ops.blend_outputs(ys, w, x=x, w_x=w_x, out_uint8=True)
    assert torch.equal(f, rf) and torch.equal(u, ru)
    # per-image weights [N, S, 1, 1]: image n is blend_outputs of image n with row n's weights
    pw = torch.tensor([[0.1, 0.6, 0.3], [0.7, 0.2, 0.1]])
    got = ops.blend_maps(ys, pw.view(N, S, 1, 1).to(DEV))
    for n in range(N):
        assert torch.equal(got[n:n + 1], ops.blend_outputs([y[n:n + 1] for y in ys], pw[n].tolist()))


def test_hard_mask_selects_styles():
    from multi_style_transfer_gan_b200 import ops
    N, C, H, W = 2, 3, 16, 32
    ys = [rand(N, C, H, W, seed=s).to(DEV) for s in range(2)]
    m = torch.zeros(1, 2, H, W, device=DEV)
    m[:, 0, :, :W // 2] = 1
    m[:, 1, :, W // 2:] = 1
    out = ops.blend_maps(ys, m)
    assert torch.equal(out[..., :W // 2], ys[0][..., :W // 2])
    assert torch.equal(out[..., W // 2:], ys[1][..., W // 2:])


@pytest.mark.parametrize("hw", [(1, 1), (3, 50), (64, 48), (17, 300)])
@pytest.mark.parametrize("sigma", [0.0, 0.5, 2.0, 6.3])
def test_gaussian_blur_matches_oracle(hw, sigma):
    from multi_style_transfer_gan_b200 import ops
    from tests import blend_maps_oracle as BM
    planes = rand(2, 3, *hw, seed=4, lo=0.0, hi=1.0)
    got = ops.gaussian_blur(planes.to(DEV), sigma).cpu()
    assert float((got.double() - BM.gaussian_blur(planes, sigma)).abs().max()) <= 1e-6
    if sigma == 0.0:
        assert torch.equal(got, planes)


def test_gaussian_blur_rejects_large_radius():
    from multi_style_transfer_gan_b200 import _lib, ops
    planes = torch.rand(1, 1, 8, 8, device=DEV)
    ops.gaussian_blur(planes, 63.7)                              # radius 255
    with pytest.raises(_lib.MsgError):
        ops.gaussian_blur(planes, 64.0)                          # radius 256
    with pytest.raises(_lib.MsgError):
        ops.gaussian_blur(planes, -1.0)


def test_blend_maps_rejects_bad_shapes():
    from multi_style_transfer_gan_b200 import _lib, ops
    ys = [torch.zeros(2, 3, 8, 8, device=DEV) for _ in range(2)]
    for maps in (torch.zeros(1, 4, 2, 2), torch.zeros(3, 2, 2, 2), torch.zeros(1, 2, 9, 8)):
        with pytest.raises(_lib.MsgError):
            ops.blend_maps(ys, maps.to(DEV))
    with pytest.raises(_lib.MsgError):                           # K = S+1 without x
        ops.blend_maps(ys, torch.zeros(1, 3, 2, 2, device=DEV))


# ---- MultiStyleStylizer ----------------------------------------------------------------------------------------------------
def make_gens(c, nb=1, S=3):
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    gens = []
    for s in range(S):
        torch.manual_seed(s)
        gens.append(EnhancedGenerator(channels=c, num_transformer_blocks=nb).to(DEV))
    return gens


def test_stylizer_constant_maps_equal_global_weights():
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    gens = make_gens(16)
    w = [0.2, 0.3, 0.5]
    x = rand(3, 3, 64, 64, seed=7).to(DEV)
    cm = torch.tensor(w).view(1, 3, 1, 1)
    cmx = torch.tensor(w + [0.25]).view(1, 4, 1, 1)
    for sched in (dict(style_streams=False, use_graph=False), dict(style_streams=True, use_graph=False),
                  dict(style_streams=True, use_graph=True)):
        st = MultiStyleStylizer(gens, micro_batch=2, **sched)
        ref = st(x, w, gain=1.1, clip=(-1, 1))
        assert torch.equal(st(x, weight_maps=cm, gain=1.1, clip=(-1, 1)), ref), sched
        assert torch.equal(st(x, weight_maps=cmx), st(x, w, w_x=0.25)), sched
        assert torch.equal(st(x, weight_maps=cm, out_uint8=True), st(x, w, out_uint8=True)), sched


def test_stylizer_maps_graph_replay_and_per_image():
    """c = 64: a second graph call with other map values replays the captured graph and equals the serial schedule; per-image
    maps through micro-batches of 2 equal one call per image; host maps equal device maps."""
    from multi_style_transfer_gan_b200 import _lib
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    gens = make_gens(64, nb=3)
    x = rand(3, 3, 64, 64, seed=8).to(DEV)
    serial = MultiStyleStylizer(gens, micro_batch=2, style_streams=False, use_graph=False)
    graph = MultiStyleStylizer(gens, micro_batch=2, style_streams=True, use_graph=True)
    maps_a = rand(3, 4, 16, 16, seed=30, lo=0.0, hi=1.0)
    maps_b = rand(3, 4, 16, 16, seed=31, lo=0.0, hi=1.0)
    ya = graph(x, weight_maps=maps_a.to(DEV), normalize_maps=True)
    n_graphs = len(graph._graphs)
    yb = graph(x, weight_maps=maps_b.to(DEV), normalize_maps=True)
    assert len(graph._graphs) == n_graphs, "new map values re-captured the graph"
    assert torch.equal(ya, serial(x, weight_maps=maps_a.to(DEV), normalize_maps=True))
    assert torch.equal(yb, serial(x, weight_maps=maps_b.to(DEV), normalize_maps=True))
    assert not torch.equal(ya, yb)
    for n in range(3):
        single = serial(x[n:n + 1].contiguous(), weight_maps=maps_a[n:n + 1].to(DEV), normalize_maps=True)
        assert torch.equal(single, ya[n:n + 1]), n
    assert torch.equal(serial(x, weight_maps=maps_a, normalize_maps=True), ya)          # host maps
    # the global-weight path launches what it launched before: S forwards and one msg_blend_outputs per micro-batch
    l0 = _lib.launches
    serial(x, [0.2, 0.3, 0.5])
    n_global = _lib.launches - l0
    l0 = _lib.launches
    serial(x, weight_maps=maps_a.to(DEV))
    assert _lib.launches - l0 == n_global


def test_stylizer_feathered_maps():
    from multi_style_transfer_gan_b200 import ops
    from multi_style_transfer_gan_b200.stylize import MultiStyleStylizer
    from tests import blend_maps_oracle as BM
    gens = make_gens(16)
    x = rand(2, 3, 64, 64, seed=9).to(DEV)
    maps = torch.zeros(2, 3, 32, 32)
    maps[:, 0, :16] = 1
    maps[:, 1, 16:] = 1
    maps[1, 2] = 0.5
    st = MultiStyleStylizer(gens, micro_batch=2, use_graph=False)
    y = st(x, weight_maps=maps, feather_sigma=3.0, normalize_maps=True)
    with torch.no_grad():
        singles = [g(x) for g in st.generators]
    ref = ops.blend_maps(singles, BM.gaussian_blur(maps, 3.0).float().to(DEV), normalize=True)
    assert float((y - ref).abs().max()) <= 1e-6
