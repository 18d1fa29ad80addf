"""Pins oracle/restate.py (the CPU oracle) against the golden vectors produced from the
unmodified reference by oracle/make_golden.py.  CPU only."""
import torch

from oracle import restate as R
from tests.util import assert_parity

TOL = dict(rtol=1e-4, atol=2e-6)
GRAD_REL = 1e-2


def synth_images(B, H, W, seed=1234):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, 3, H, W, generator=g) * 2 - 1


def test_generator_forward_and_grads(golden):
    g = golden("gen_c16_b1_64x48.pt")
    assert g["keys"] == R.generator_state_dict_keys()
    assert g["children"] == ["initial", "down1", "down2", "transformer_blocks", "up1", "up2",
                             "output", "style_encoder"]
    sd = {k: v.clone().requires_grad_(True) for k, v in g["state_dict"].items()}
    x = g["x"].clone().requires_grad_(True)
    y = R.generator_forward(sd, x)
    assert_parity(y, g["y"], 1e-4, "y")
    loss = (y * g["r"]).sum() / y.numel() + ((y - g["r"]) ** 2).mean()
    torch.testing.assert_close(loss, g["loss"], **TOL)
    grads = torch.autograd.grad(loss, [x] + list(sd.values()), allow_unused=True)
    check_generator_grads(g, grads[0], dict(zip(sd.keys(), grads[1:])))


def check_generator_grads(g, dx, grads, rel=GRAD_REL):
    """fp32 gradient noise floor: the reference's own fp32 grads differ from an fp64 evaluation of
    the same graph by 1e-3..4e-3 (normalised max) per tensor (measured, DESIGN.md), so gradients
    are compared at GRAD_REL = 1e-2, not 1e-4.  Conv biases that feed an InstanceNorm have an
    analytically-zero gradient (|g| ~ 1e-8 of pure rounding noise in the reference): they are
    checked to be ~0 against the global gradient scale instead."""
    gmax = max(float(v.abs().max()) for v in g["grads"].values() if v is not None)
    assert_parity(dx, g["dx"], rel, "dx")
    for k, ref in g["grads"].items():
        gr = grads[k]
        if ref is None:  # style_encoder: dead path with identity blocks
            assert gr is None or float(gr.abs().max()) == 0.0, k
            continue
        if float(ref.abs().max()) < 1e-5 * gmax:
            assert float(gr.abs().max()) < 1e-4 * gmax, k
            continue
        assert_parity(gr, ref, rel, k)


def test_blocks(golden):
    g = golden("blocks_c32.pt")
    la = g["local_attention"]
    sd = la["state_dict"]
    y = R.local_attention(la["x"], sd["qkv.weight"], sd["qkv.bias"], sd["proj.weight"], sd["proj.bias"])
    assert_parity(y, la["y"], 1e-4, "la")
    msb = g["multi_scale_block"]
    y = R.multi_scale_block(msb["x"], {f"m.{k}": v for k, v in msb["state_dict"].items()}, "m")
    assert_parity(y, msb["y"], 1e-4, "msb")


def test_bad_size_raises():
    import pytest
    sd = {}
    with pytest.raises(RuntimeError):
        R.generator_forward(sd, torch.zeros(1, 3, 130, 130))


def test_discriminator(golden):
    g = golden("disc_c8_64.pt")
    sd = {k: v.clone() for k, v in g["state_dict_before"].items()}
    for k in sd:
        if k.endswith("weight_orig") or k.endswith("bias"):
            sd[k].requires_grad_(True)
    x = g["x"].clone().requires_grad_(True)
    score, struct, new_uv = R.discriminator_forward(sd, x, training=True)
    torch.testing.assert_close(score, g["score"], **TOL)
    torch.testing.assert_close(struct, g["struct"], **TOL)
    for name, (u, v) in new_uv.items():
        torch.testing.assert_close(u, g["state_dict_after"][f"{name}.weight_u"], **TOL)
        torch.testing.assert_close(v, g["state_dict_after"][f"{name}.weight_v"], **TOL)
    loss = ((score - 1) ** 2).mean() + struct.abs().mean()
    names = [k for k in sd if sd[k].requires_grad]
    grads = torch.autograd.grad(loss, [x] + [sd[k] for k in names])
    check_generator_grads(g, grads[0], dict(zip(names, grads[1:])))
    e = golden("disc_c8_64_eval_b1.pt")
    sd_after = g["state_dict_after"]
    s1, st1, _ = R.discriminator_forward(sd_after, synth_images(1, 64, 64), training=False)
    assert list(s1.shape) == e["score_shape"] == []  # .squeeze() -> 0-dim at B=1
    torch.testing.assert_close(s1, e["score"], **TOL)
    torch.testing.assert_close(st1, e["struct"], **TOL)


def test_train_step(golden):
    g = golden("train_step_c8_64.pt")
    m = R.OracleCycleGAN(g["init"]["G_AB"], g["init"]["G_BA"], g["init"]["D_A"], g["init"]["D_B"])
    # step 1: <=1e-4 relative.  step 2 sees weights after Adam's first update, which is
    # lr*g/(|g|+eps) ~ lr*sign(g): fp32 gradient noise is amplified (sign flips of ~0 grads), the
    # reference vs its own restatement already differ by 2.4e-4 there -> 2e-3 for step 2.
    for step, ref in enumerate(g["losses"]):
        got = m.train_step(g["real_A"], g["real_B"])
        tol = 1e-4 if step == 0 else 2e-3
        for k in ref:
            assert abs(got[k] - ref[k]) <= tol * abs(ref[k]) + 1e-6, (step, k, got[k], ref[k])
    # spectral-norm buffers advanced by 10 power iterations per step, in the reference's order
    for n in ("D_A", "D_B"):
        for k, v in g["final"][n].items():
            if k.endswith("weight_u") or k.endswith("weight_v"):
                assert_parity(getattr(m, n)[k], v, 2e-3, f"{n}.{k}")


def test_config1_blend(golden):
    for c in (16,):
        g = golden(f"config1_c{c}_256.pt")
        ref = R.blend_outputs([g["y0"], g["y1"]], g["w"])
        assert ref.shape == (1, 3, 256, 256)
        assert float(ref.abs().max()) <= 1.0


def test_gram_properties():
    torch.manual_seed(0)
    f = torch.relu(torch.randn(2, 8, 5, 7))
    G = R.gram(f)
    torch.testing.assert_close(G, G.transpose(1, 2))
    assert (torch.linalg.eigvalsh(G.double()) > -1e-9).all()
    assert float(R.style_loss([f], [f])) == 0.0


def test_pretrain_generator(golden):
    """oracle restatement of pretrain.Generator (BatchNorm auto-encoder) against the golden from the unmodified
    reference: train-mode forward, running-statistics update, masked-L1 loss and its gradients, eval-mode forward."""
    g = golden("pretrain_c8_64.pt")
    sd = {k: v.clone() for k, v in g["init"].items()}
    params = {k: v.requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
    sd.update(params)
    x = g["masked"].clone().requires_grad_(True)
    y, new = R.pretrain_generator_forward(sd, x, training=True)
    assert_parity(y, g["y_train"], 1e-6, "pretrain y (train mode)")
    loss = R.pretrain_masked_l1(y, g["real"], g["mask"])
    assert abs(float(loss) - float(g["loss"])) <= 1e-6
    loss.backward()
    # the conv biases in front of each BatchNorm have an analytically-zero gradient (~1e-10 of rounding noise in the
    # reference, which the summation order of the host's CPU changes): check_generator_grads tests them for ~0
    check_generator_grads(g, x.grad, {k: p.grad for k, p in params.items()}, rel=1e-4)
    for k, ref in g["running_after"].items():
        assert torch.allclose(new[k].double(), ref.double(), rtol=1e-6, atol=1e-7), k
    sd2 = {k: v.detach() for k, v in sd.items()}
    sd2.update(g["running_after"])
    y_eval, _ = R.pretrain_generator_forward(sd2, g["masked"], training=False)
    assert_parity(y_eval, g["y_eval"], 1e-6, "pretrain y (eval mode)")
