"""The reference's own import lines resolve against dropin/ (the shim directory a maintainer puts first on sys.path,
INTEGRATION.md).  CPU only: construction and state_dict layout, no kernels."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r"""
import sys
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
# enhanced_train.py:10-11, batch_process_images.py:18, m_test.py:12, enhanced_generator.py:4 of the reference
from enhanced_generator import EnhancedGenerator, EnhancedDiscriminator
from pretrain import MonetPhotoDataset, set_seed
from pretrain import Generator
from structural_transformer import StructuralTransformerBlock
from enhanced_train import EnhancedCycleGAN
import enhanced_generator, multi_style_transfer_gan_b200.enhanced_generator as ours
assert enhanced_generator.EnhancedGenerator is ours.EnhancedGenerator
set_seed(1)
g = EnhancedGenerator(16, 1)
keys = list(g.state_dict().keys())
assert keys[0] == 'initial.0.weight' and g.state_dict()[keys[0]].shape[0] == 16     # direct_transform.py:25-28 reads this
assert [n for n, _ in g.named_children()] == ['initial', 'down1', 'down2', 'transformer_blocks', 'up1', 'up2', 'output', 'style_encoder']
d = EnhancedDiscriminator(16)
assert len(d.state_dict()) == 28
import tempfile, os
root = tempfile.mkdtemp(); os.makedirs(os.path.join(root, 'trainA'))
assert len(MonetPhotoDataset(root, 'A')) == 0
print('dropin ok')
"""


def test_reference_import_lines_resolve_against_dropin():
    r = subprocess.run([sys.executable, "-c", SCRIPT, ROOT, os.path.join(ROOT, "dropin")], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "dropin ok" in r.stdout


LOAD_MODELS_SCRIPT = r"""
import os, sys, tempfile
root, dropin, ref = sys.argv[1:4]
sys.path.insert(0, ref); sys.path.insert(0, root); sys.path.insert(0, dropin)      # dropin/ first: it shadows the reference modules
import torch
from enhanced_generator import EnhancedGenerator
import multi_style_transfer_gan_b200.enhanced_generator as ours
# checkpoints in the layout EnhancedCycleGAN.save_models writes (enhanced_train.py:133-152)
work = tempfile.mkdtemp(); os.makedirs(os.path.join(work, 'models')); os.chdir(work)
torch.manual_seed(0); a = EnhancedGenerator(16, 1)
torch.manual_seed(1); b = EnhancedGenerator(16, 1)
torch.save({'epoch': 200, 'G_AB_state_dict': a.state_dict()}, 'models/G_AB_epoch_200.pth')
torch.save(b.state_dict(), 'models/G_BA_epoch_200.pth')                            # the bare-dict variant (:104-108)
import batch_process_images as bpi                                                  # the UNMODIFIED reference script
assert bpi.EnhancedGenerator is ours.EnhancedGenerator                              # bound to the shim, not to the reference class
models = bpi.load_models(torch.device('cpu'))
assert set(models) == {'enhanced_AB', 'enhanced_BA'}, set(models)
for m, src in ((models['enhanced_AB'], a), (models['enhanced_BA'], b)):
    assert isinstance(m, ours.EnhancedGenerator) and not m.training
    for (k, v), (k2, v2) in zip(m.state_dict().items(), src.state_dict().items()):
        assert k == k2 and torch.equal(v, v2)
# the model call of process_cyclegan / process_enhanced (:206-209, :293-295) on a CPU tensor: this package has no CPU path and says so
try:
    with torch.no_grad():
        models['enhanced_AB'](torch.zeros(1, 3, 64, 64))
    raise SystemExit('expected an error on a CPU tensor')
except Exception as e:
    assert 'no CPU path' in str(e) or 'CPU' in str(e), repr(e)
print('load_models ok')
"""


def test_reference_load_models_runs_against_dropin():
    """batch_process_images.load_models of the UNMODIFIED reference (batch_process_images.py:60-120), imported with dropin/ first
    on sys.path: it builds OUR classes, loads both checkpoint layouts the reference writes, and the model call refuses a CPU
    tensor loudly.  Needs a checkout of the reference (oracle/ref_import.py)."""
    import pytest
    from oracle import ref_import
    if not ref_import.available():
        pytest.skip(f"no checkout of the reference at {ref_import.REFERENCE_ROOT}")
    r = subprocess.run([sys.executable, "-c", LOAD_MODELS_SCRIPT, ROOT, os.path.join(ROOT, "dropin"), ref_import.REFERENCE_ROOT],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "load_models ok" in r.stdout
