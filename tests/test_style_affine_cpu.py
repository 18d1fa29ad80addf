"""CPU: the style-conditional EnhancedGenerator's parameters, checkpoint compatibility, argument checks (no device needed) and
the CPU restatement it is checked against on the GPU (tests/style_affine_oracle.py)."""
import pytest
import torch

from multi_style_transfer_gan_b200.enhanced_generator import EnhancedGenerator
from oracle import restate as R
from tests import style_affine_oracle as O

HOLDERS = (["initial.1"] + [f"{s}.1" for s in O.STAGES] + [f"{s}.4.branch{i}.1" for s in O.STAGES for i in range(1, 5)]
           + [f"{s}.4.fusion.1" for s in O.STAGES])


def test_enable_style_affine_adds_exactly_the_affine_keys():
    torch.manual_seed(0)
    G = EnhancedGenerator(16, 1)
    plain = list(G.state_dict().keys())
    rng = torch.get_rng_state()
    assert G.enable_style_affine(3) is G
    assert torch.equal(rng, torch.get_rng_state())
    keys = list(G.state_dict().keys())
    assert len(HOLDERS) == 25 and len(plain) == 70
    added = [k for k in keys if k not in plain]
    assert sorted(added) == sorted(f"{h}.{p}" for h in HOLDERS for p in ("weight", "bias"))
    it = iter(keys)
    assert all(k in it for k in plain)                      # the plain keys, in their order
    assert keys[0] == "initial.0.weight"
    sd = G.state_dict()
    for h in HOLDERS:
        C = G.get_submodule(h).num_features
        assert sd[f"{h}.weight"].shape == (3, C) and torch.equal(sd[f"{h}.weight"], torch.ones(3, C))
        assert sd[f"{h}.bias"].shape == (3, C) and torch.equal(sd[f"{h}.bias"], torch.zeros(3, C))
    # the seeded init of the plain parameters is untouched
    torch.manual_seed(0)
    ref = EnhancedGenerator(16, 1).state_dict()
    assert all(torch.equal(ref[k], sd[k]) for k in plain)


def test_plain_checkpoint_loads_into_conditional_model():
    plain = EnhancedGenerator(16, 1).state_dict()
    G = EnhancedGenerator(16, 1).enable_style_affine(2)
    res = G.load_state_dict(plain, strict=False)
    assert sorted(res.missing_keys) == sorted(f"{h}.{p}" for h in HOLDERS for p in ("weight", "bias"))
    assert res.unexpected_keys == []


def test_style_argument_errors_need_no_device():
    G = EnhancedGenerator(8, 1).enable_style_affine(3)
    x = torch.zeros(2, 3, 32, 32)
    bad = [None, [0.5, 0.5], torch.zeros(4), torch.zeros(3, 3), torch.zeros(2, 2), torch.zeros(1, 2, 3),
           torch.zeros(3, dtype=torch.float64), torch.zeros(3, requires_grad=True), torch.zeros(2, 3, requires_grad=True)]
    for st in bad:
        with pytest.raises(ValueError):
            G(x, style=st)
    with pytest.raises(ValueError):
        EnhancedGenerator(8, 1)(x, style=[1.0])
    with pytest.raises(ValueError):
        G.enable_style_affine(3)
    with pytest.raises(ValueError):
        EnhancedGenerator(8, 1).enable_style_affine(0)


def _sd(c, S, seed):
    torch.manual_seed(seed)
    return EnhancedGenerator(c, 0).enable_style_affine(S).state_dict()


def test_oracle_identity_affine_is_the_plain_restatement():
    sd = _sd(8, 3, 1)
    x = torch.rand(2, 3, 32, 32, generator=torch.Generator().manual_seed(2)) * 2 - 1
    for s in range(3):
        w = torch.zeros(3)
        w[s] = 1
        assert torch.equal(O.generator_forward(sd, x, w), R.generator_forward(sd, x))


def test_oracle_per_image_mix_matches_blended_affine_loop():
    sd = O.random_affines(_sd(8, 3, 3), 3, seed=4)
    x = torch.rand(3, 3, 32, 32, generator=torch.Generator().manual_seed(5)) * 2 - 1
    w = torch.tensor([[0.2, 0.3, 0.5], [1.0, 0.0, 0.0], [-0.5, 1.25, 0.75]])
    y = O.generator_forward(sd, x, w)
    for n in range(3):
        yn = O.generator_forward(sd, x[n:n + 1], norm=O.blended_norm(sd, w[n]))
        torch.testing.assert_close(y[n:n + 1], yn, rtol=1e-4, atol=1e-4)     # (batched vs single-image convs)
    # a shared [S] mix is the [B, S] mix with equal rows
    assert torch.equal(O.generator_forward(sd, x, w[0]), O.generator_forward(sd, x, w[0].expand(3, 3)))
    # the affines do something
    assert (O.generator_forward(sd, x, w[1]) - O.generator_forward(sd, x, w[2])).abs().max() > 1e-2
