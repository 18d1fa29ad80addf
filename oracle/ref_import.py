"""TEST INFRASTRUCTURE ONLY -- imports the *real* reference (read-only) from a checkout of it at
``oracle/_ref/`` (kept out of git) or at ``$MSG_REFERENCE_ROOT``.

The reference cannot be imported as shipped: ``enhanced_generator.py:4`` imports
``StructuralTransformerBlock`` from a module ``structural_transformer`` that is not in the
repository (SURVEY.md F2).  This shim registers an identity stub under that name in
``sys.modules`` *before* importing, which is the only thing pinned about the block
(ctor ``StructuralTransformerBlock(dim=...)``, call ``block(x, style, orig) -> x``,
enhanced_generator.py:114-117, :222-223).

The reference is not part of this repository, so this file is used solely by
``oracle/make_golden.py`` and by the tests marked ``reference``, which skip without a checkout.
Everything else is pinned to the reference by the vectors in ``tests/golden/``.  Nothing under
``multi_style_transfer_gan_b200/`` may import it.
"""
import os
import sys
import types
import warnings

REFERENCE_ROOT = os.environ.get("MSG_REFERENCE_ROOT", os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref"))


def available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "enhanced_generator.py"))


def _install_stub():
    if "structural_transformer" in sys.modules:
        return
    import torch.nn as nn

    class StructuralTransformerBlock(nn.Module):
        """Identity stand-in for the missing block (interface only; parity unpinned)."""

        def __init__(self, dim):
            super().__init__()
            self.dim = dim

        def forward(self, x, style, orig_input):
            return x

    mod = types.ModuleType("structural_transformer")
    mod.StructuralTransformerBlock = StructuralTransformerBlock
    sys.modules["structural_transformer"] = mod


def load():
    """Returns (enhanced_generator, enhanced_train) modules of the unmodified reference."""
    if not available():
        raise RuntimeError(f"reference not present at {REFERENCE_ROOT}")
    _install_stub()
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        import enhanced_generator as eg  # noqa: E402
        import enhanced_train as et  # noqa: E402
    return eg, et
