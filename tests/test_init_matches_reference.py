"""The drop-in classes must consume the RNG exactly like the reference's constructors, so
`torch.manual_seed(s); Model(...)` yields bit-identical parameters and buffers (this is what lets
goldens for the c=64 model be stored without their 10 MB of weights).

The `*_matches_stored_reference` tests compare against the reference's own seeded state dicts that
oracle/make_golden.py stored in tests/golden/, and test_seeded_generator_reproduces_stored_reference_outputs
against its stored c=16 and c=64 outputs; the tests marked `reference` import a checkout of the
reference itself (oracle/ref_import.py) and cover further seeds and sizes."""
import pytest
import torch


def _assert_same_state(ref_sd, mine, name=""):
    ms = mine.state_dict()
    assert list(ref_sd.keys()) == list(ms.keys()), name
    for k in ref_sd:
        assert torch.equal(ref_sd[k], ms[k]), (name, k)


def _assert_same_init(ref_sd, ref_param_names, mine):
    _assert_same_state(ref_sd, mine)
    assert list(ref_param_names) == [n for n, _ in mine.named_parameters()]
    mine.load_state_dict(ref_sd, strict=True)


def test_generator_init_matches_stored_reference(golden):
    """EnhancedGenerator(16, 1) after manual_seed(0), as stored with the reference's forward and gradients (grads keep the
    order of named_parameters)."""
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    g = golden("gen_c16_b1_64x48.pt")
    torch.manual_seed(0)
    mine = EnhancedGenerator(channels=16, num_transformer_blocks=1)
    _assert_same_init(g["state_dict"], g["grads"].keys(), mine)
    assert g["children"] == [n for n, _ in mine.named_children()]


def test_discriminator_init_matches_stored_reference(golden):
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedDiscriminator
    g = golden("disc_c8_64.pt")
    torch.manual_seed(0)
    _assert_same_init(g["state_dict_before"], g["grads"].keys(), EnhancedDiscriminator(channels=8))


def test_cyclegan_members_init_matches_stored_reference(golden):
    """The reference's train-step golden builds G_AB, G_BA (c=8, 1 block), D_A, D_B (c=8) in this order after manual_seed(7):
    one RNG stream through four constructors."""
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedDiscriminator, EnhancedGenerator
    init = golden("train_step_c8_64.pt")["init"]
    torch.manual_seed(7)
    for name, mine in (("G_AB", EnhancedGenerator(channels=8, num_transformer_blocks=1)),
                       ("G_BA", EnhancedGenerator(channels=8, num_transformer_blocks=1)),
                       ("D_A", EnhancedDiscriminator(channels=8)), ("D_B", EnhancedDiscriminator(channels=8))):
        _assert_same_state(init[name], mine, name)


def test_pretrain_generator_init_matches_stored_reference(golden):
    """pretrain.Generator(channels=8) after manual_seed(0), BatchNorm buffers included."""
    from multi_style_transfer_gan_b200.pretrain import Generator
    g = golden("pretrain_c8_64.pt")
    torch.manual_seed(0)
    _assert_same_init(g["init"], g["grads"].keys(), Generator(channels=8))


@pytest.mark.parametrize("c,nb", [(16, 1), (64, 3)])
def test_seeded_generator_reproduces_stored_reference_outputs(golden, c, nb):
    """The c=64 goldens keep the reference's outputs, not its weights: our EnhancedGenerator(c, nb) after manual_seed(seed),
    run through the CPU oracle, must give the reference's stored forward of the same seed (an init drawn in any other order
    misses by O(1)).  Covers the benchmarked c=64 / 3-block model and restate.py on a generator with several blocks.
    Tolerances as in test_gpu_models.test_config1_two_style_blend (the reference's own fp32 noise floor at c=64)."""
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    from oracle import restate as R
    from tests.util import assert_parity
    g = golden(f"config1_c{c}_256.pt")
    x = torch.rand(1, 3, 256, 256, generator=torch.Generator().manual_seed(g["x_seed"])) * 2 - 1
    for seed, key in zip(g["seeds"], ("y0", "y1")):
        torch.manual_seed(seed)
        sd = {k: v.detach() for k, v in EnhancedGenerator(channels=c, num_transformer_blocks=nb).state_dict().items()}
        with torch.no_grad():
            y = R.generator_forward(sd, x)
        assert_parity(y, g[key], 1e-4, f"seed {seed}", max_rel=1e-4 if c == 16 else 5e-4)


@pytest.mark.reference
@pytest.mark.parametrize("c,nb", [(16, 1), (64, 3), (8, 2)])
def test_generator_init_bit_identical(c, nb):
    from oracle import ref_import
    eg, _ = ref_import.load()
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
    torch.manual_seed(5)
    ref = eg.EnhancedGenerator(channels=c, num_transformer_blocks=nb)
    torch.manual_seed(5)
    mine = EnhancedGenerator(channels=c, num_transformer_blocks=nb)
    rs, ms = ref.state_dict(), mine.state_dict()
    assert list(rs.keys()) == list(ms.keys())
    for k in rs:
        assert torch.equal(rs[k], ms[k]), k
    assert [n for n, _ in ref.named_children()] == [n for n, _ in mine.named_children()]
    assert [n for n, _ in ref.named_parameters()] == [n for n, _ in mine.named_parameters()]
    mine.load_state_dict(rs, strict=True)   # convert_model.py / pth_info.py contract: strict round trip
    ref.load_state_dict(ms, strict=True)


@pytest.mark.reference
@pytest.mark.parametrize("c", [16, 8])
def test_discriminator_init_bit_identical(c):
    from oracle import ref_import
    eg, _ = ref_import.load()
    from multi_style_transfer_gan_b200.enhanced_generator import EnhancedDiscriminator
    torch.manual_seed(9)
    ref = eg.EnhancedDiscriminator(channels=c)
    torch.manual_seed(9)
    mine = EnhancedDiscriminator(channels=c)
    rs, ms = ref.state_dict(), mine.state_dict()
    assert list(rs.keys()) == list(ms.keys())
    for k in rs:
        assert torch.equal(rs[k], ms[k]), k
    assert [n for n, _ in ref.named_parameters()] == [n for n, _ in mine.named_parameters()]
    ref.load_state_dict(ms, strict=True)
    mine.load_state_dict(rs, strict=True)


@pytest.mark.reference
def test_oracle_restatement_matches_live_reference():
    """restate.py vs the imported reference on fresh random weights (not only the goldens)."""
    from oracle import ref_import, restate as R
    from tests.util import assert_parity
    eg, _ = ref_import.load()
    torch.manual_seed(21)
    ref = eg.EnhancedGenerator(channels=8, num_transformer_blocks=2).eval()
    x = torch.rand(1, 3, 32, 48) * 2 - 1
    with torch.no_grad():
        assert_parity(R.generator_forward(dict(ref.state_dict()), x), ref(x), 1e-4, "G")
    D = eg.EnhancedDiscriminator(channels=8).eval()
    x = torch.rand(3, 3, 64, 64) * 2 - 1
    with torch.no_grad():
        s, st = D(x)
        s2, st2, _ = R.discriminator_forward(dict(D.state_dict()), x, training=False)
    assert_parity(s2, s, 1e-4, "score")
    assert_parity(st2, st, 1e-4, "struct")


@pytest.mark.reference
@pytest.mark.parametrize("c", [64, 8])
def test_pretrain_generator_init_bit_identical(c):
    """pretrain.Generator (pretrain.py:60-97): same module tree, state_dict keys (incl. BatchNorm buffers) and default
    init in the same RNG order."""
    import importlib
    from oracle import ref_import
    ref_import.load()
    pt = importlib.import_module("pretrain")
    from multi_style_transfer_gan_b200.pretrain import Generator
    torch.manual_seed(3)
    ref = pt.Generator(channels=c)
    torch.manual_seed(3)
    mine = Generator(channels=c)
    rs, ms = ref.state_dict(), mine.state_dict()
    assert list(rs.keys()) == list(ms.keys())
    for k in rs:
        assert torch.equal(rs[k], ms[k]), k
    assert [n for n, _ in ref.named_parameters()] == [n for n, _ in mine.named_parameters()]
    mine.load_state_dict(rs, strict=True)
    ref.load_state_dict(ms, strict=True)
