"""TEST INFRASTRUCTURE ONLY -- generates tests/golden/*.pt from the UNMODIFIED reference.

Run with a checkout of the reference at oracle/_ref/ (or $MSG_REFERENCE_ROOT):  python oracle/make_golden.py
The reference has no tests, fixtures or checkpoints of its own (SURVEY.md section 4), so the golden
vectors are outputs of the reference classes themselves: seeded random init
(torch.manual_seed(seed) before the constructor), seeded synthetic input
(torch.manual_seed(1234); rand*2-1), fp32, CPU.  Files stay small: weights are stored only for
the small models; for the c=64 config-1 case the weights are re-created from the seed by the
product's own constructor (tests/test_init_matches_reference.py pins that the two inits are
bit-identical) or by the oracle-side helper below.
"""
import os
import sys
import warnings

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
from oracle import ref_import  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), "tests", "golden")


def synth_images(B, H, W, seed=1234):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(B, 3, H, W, generator=g) * 2 - 1


def build(cls, seed, *a, **k):
    torch.manual_seed(seed)
    return cls(*a, **k)


def main():
    warnings.simplefilter("ignore")
    torch.set_num_threads(os.cpu_count())
    eg, et = ref_import.load()
    os.makedirs(OUT, exist_ok=True)

    # ---- G small: c=16 / 1 block (the size the reference trains and deploys), fwd + all grads
    G = build(eg.EnhancedGenerator, 0, channels=16, num_transformer_blocks=1)
    x = synth_images(2, 64, 48)
    x.requires_grad_(True)
    y = G(x)
    r = synth_images(2, 64, 48, seed=99)
    loss = (y * r).sum() / y.numel() + ((y - r) ** 2).mean()
    loss.backward()
    torch.save({
        "state_dict": {k: v.detach().clone() for k, v in G.state_dict().items()},
        "x": x.detach(), "y": y.detach(), "r": r, "loss": loss.detach(),
        "dx": x.grad.clone(),
        "grads": {k: (p.grad.clone() if p.grad is not None else None) for k, p in G.named_parameters()},
        "keys": list(G.state_dict().keys()),
        "children": [n for n, _ in G.named_children()],
    }, os.path.join(OUT, "gen_c16_b1_64x48.pt"))

    # ---- config 1: [1,3,256,256], two state dicts (seeds 0, 1), blend 0.7/0.3 ; c=16 and c=64
    x = synth_images(1, 256, 256)
    for c, nb in ((16, 1), (64, 3)):
        ys = []
        with torch.no_grad():
            for seed in (0, 1):
                ys.append(build(eg.EnhancedGenerator, seed, channels=c, num_transformer_blocks=nb).eval()(x))
        blend = 0.7 * ys[0] + 0.3 * ys[1]
        torch.save({"y0": ys[0], "y1": ys[1], "w": [0.7, 0.3], "seeds": [0, 1],
                    "x_seed": 1234}, os.path.join(OUT, f"config1_c{c}_256.pt"))

    # ---- D small: c=8, training-mode forward (power iteration), grads
    D = build(eg.EnhancedDiscriminator, 0, channels=8)
    sd0 = {k: v.detach().clone() for k, v in D.state_dict().items()}
    x = synth_images(2, 64, 64)
    x.requires_grad_(True)
    score, struct = D(x)
    loss = ((score - 1) ** 2).mean() + struct.abs().mean()
    loss.backward()
    sd1 = {k: v.detach().clone() for k, v in D.state_dict().items()}
    torch.save({"state_dict_before": sd0, "state_dict_after": sd1, "x": x.detach(),
                "score": score.detach(), "struct": struct.detach(), "loss": loss.detach(),
                "dx": x.grad.clone(),
                "grads": {k: p.grad.clone() for k, p in D.named_parameters()},
                "keys": list(sd0.keys())}, os.path.join(OUT, "disc_c8_64.pt"))
    # B=1 squeeze quirk (0-dim score), eval mode (no power iteration)
    D.eval()
    with torch.no_grad():
        s1, st1 = D(synth_images(1, 64, 64))
    torch.save({"score_shape": list(s1.shape), "score": s1, "struct": st1},
               os.path.join(OUT, "disc_c8_64_eval_b1.pt"))

    # ---- train_step: the real EnhancedCycleGAN, shrunk to c=8 by re-building its members
    torch.manual_seed(0)
    m = et.EnhancedCycleGAN()  # constructs c=16 nets on CPU; replace with c=8 ones for file size
    import itertools
    import torch.optim as optim
    torch.manual_seed(7)
    m.G_AB = eg.EnhancedGenerator(channels=8, num_transformer_blocks=1)
    m.G_BA = eg.EnhancedGenerator(channels=8, num_transformer_blocks=1)
    m.D_A = eg.EnhancedDiscriminator(channels=8)
    m.D_B = eg.EnhancedDiscriminator(channels=8)
    m.G_AB.gradient_checkpointing_enable()
    m.G_BA.gradient_checkpointing_enable()
    m.g_optimizer = optim.Adam(itertools.chain(m.G_AB.parameters(), m.G_BA.parameters()),
                               lr=5e-5, betas=(0.5, 0.999))
    m.d_optimizer = optim.Adam(itertools.chain(m.D_A.parameters(), m.D_B.parameters()),
                               lr=2e-4, betas=(0.5, 0.999))
    init = {n: {k: v.detach().clone() for k, v in getattr(m, n).state_dict().items()}
            for n in ("G_AB", "G_BA", "D_A", "D_B")}
    real_A = synth_images(2, 64, 64, seed=11)
    real_B = synth_images(2, 64, 64, seed=12)
    losses = [m.train_step(real_A, real_B) for _ in range(2)]
    final = {n: {k: v.detach().clone() for k, v in getattr(m, n).state_dict().items()}
             for n in ("G_AB", "G_BA", "D_A", "D_B")}
    torch.save({"init": init, "final": final, "losses": losses, "real_A": real_A, "real_B": real_B},
               os.path.join(OUT, "train_step_c8_64.pt"))

    # ---- LocalAttention / MultiScaleBlock module-level vectors (layer-wise bisecting)
    torch.manual_seed(3)
    la = eg.LocalAttention(32, window_size=4)
    msb = eg.MultiScaleBlock(32)
    xa = torch.randn(2, 32, 16, 24)
    xa.requires_grad_(True)
    ya = la(xa)
    ya.square().mean().backward()
    la_pack = {"state_dict": {k: v.detach().clone() for k, v in la.state_dict().items()},
               "x": xa.detach().clone(), "y": ya.detach(), "dx": xa.grad.clone(),
               "grads": {k: p.grad.clone() for k, p in la.named_parameters()}}
    xb = torch.randn(2, 32, 16, 24)
    xb.requires_grad_(True)
    yb = msb(xb)
    yb.square().mean().backward()
    msb_pack = {"state_dict": {k: v.detach().clone() for k, v in msb.state_dict().items()},
                "x": xb.detach().clone(), "y": yb.detach(), "dx": xb.grad.clone(),
                "grads": {k: p.grad.clone() for k, p in msb.named_parameters()}}
    torch.save({"local_attention": la_pack, "multi_scale_block": msb_pack},
               os.path.join(OUT, "blocks_c32.pt"))

    # ---- pretrain.Generator (BatchNorm auto-encoder, pretrain.py:60-97) + the masked-L1 objective (:159-160)
    import pretrain as pt  # the unmodified reference module (imports cleanly once the stub is installed)
    Gp = build(pt.Generator, 0, channels=8)
    init = {k: v.detach().clone() for k, v in Gp.state_dict().items()}
    real = synth_images(3, 64, 64, seed=21)
    gm = torch.Generator().manual_seed(22)
    mask = (torch.rand(3, 1, 64, 64, generator=gm) > 0.3).float()
    masked = (real * mask).requires_grad_(True)
    Gp.train()
    y = Gp(masked)
    loss = torch.nn.L1Loss()(y * (1 - mask), real * (1 - mask))
    loss.backward()
    after = {k: v.detach().clone() for k, v in Gp.state_dict().items() if "running" in k or "num_batches" in k}
    Gp.eval()
    with torch.no_grad():
        y_eval = Gp(masked.detach())
    torch.save({"init": init, "real": real, "mask": mask, "masked": masked.detach().clone(), "y_train": y.detach(),
                "loss": loss.detach(), "dx": masked.grad.clone(),
                "grads": {k: p.grad.clone() for k, p in Gp.named_parameters()},
                "running_after": after, "y_eval": y_eval, "keys": list(Gp.state_dict().keys())},
               os.path.join(OUT, "pretrain_c8_64.pt"))

    for f in sorted(os.listdir(OUT)):
        print(f, os.path.getsize(os.path.join(OUT, f)))


if __name__ == "__main__":
    main()
