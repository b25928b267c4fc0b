"""CPU: the drop-in contract against the reference's parameter surface — state_dicts cross-load strictly in both
directions for every variant, and the reference's own `train.py`-style builder loop (`_build_lit`, train.py:1251-1271:
call the zero-arg builder, else try (num_classes, lr) / (num_classes) / ()) works on this tree's VARIANTS. No compute
runs (there is no CPU path); this is registry + parameter-surface parity.

The reference's state_dict of each variant (keys in order, shapes) is the one stored in tests/golden/init_seed42.npz
and tests/golden/cicek_init_seed42.npz, written from the reference's own constructors by oracle/make_golden.py and
oracle/make_golden_3dunet.py. Those files do not record dtypes: the dtypes the test expects (fp32, int64 for
BatchNorm's `num_batches_tracked`) are PyTorch's defaults for these modules, an assumption of the test rather than a
comparison with the reference."""
import os

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
VARIANTS = ["SPFF-UNet", "E_SP_UNet", "FG_SP_UNet", "SP_UNet", "PlainCore_UNet", "3DUNet"]


def reference_surface(variant):
    """[(key, shape)] of the reference's state_dict, in its order."""
    if variant == "3DUNet":
        z = np.load(os.path.join(GOLD, "cicek_init_seed42.npz"))
        return [(k, tuple(int(v) for v in z[k][:-2])) for k in z.files]
    z = np.load(os.path.join(GOLD, "init_seed42.npz"))
    return [(k.split("|", 1)[1], tuple(int(v) for v in z[k][:-2])) for k in z.files if k.split("|", 1)[0] == variant]


def reference_state_dict(variant, seed):
    """A state_dict with the reference's keys, order and shapes; fp32 values (BatchNorm's step counter: int64)."""
    g = torch.Generator().manual_seed(seed)
    return {k: torch.randint(0, 1000, shape, generator=g, dtype=torch.int64) if k.endswith("num_batches_tracked")
            else torch.randn(shape, generator=g) for k, shape in reference_surface(variant)}


def _mine():
    from innovative3D import config as C
    return dict((v[0], v[1]) for v in C.VARIANTS)


@pytest.mark.parametrize("variant", VARIANTS)
def test_state_dicts_cross_load(variant):
    sd_ref = reference_state_dict(variant, seed=1)
    torch.manual_seed(2)
    mine = _mine()[variant]()
    sd_mine = mine.state_dict()
    assert list(sd_ref) == list(sd_mine)                       # same keys in the same order
    assert all(sd_ref[k].shape == sd_mine[k].shape and sd_ref[k].dtype == sd_mine[k].dtype for k in sd_ref)
    mine.load_state_dict(sd_ref, strict=True)
    assert all(torch.equal(mine.state_dict()[k], sd_ref[k]) for k in sd_ref)
    torch.manual_seed(3)
    other = _mine()[variant]().state_dict()
    # what the reference's load_state_dict(strict=True) checks of this tree's state_dict: the same keys, the same shapes
    assert [(k, tuple(v.shape)) for k, v in other.items()] == reference_surface(variant)
    buffers = {k for k, _ in mine.named_buffers()}
    assert sum(int(np.prod(s)) for k, s in reference_surface(variant) if k not in buffers) == \
        sum(p.numel() for p in mine.parameters())


def test_train_py_builder_loop_on_this_trees_variants():
    """train.py:1251-1271 `_build_lit`, restated: a VARIANTS entry is a zero-arg factory or a class tried with
    (num_classes, lr), (num_classes), ()."""
    from innovative3D import config as C

    def build_lit(builder):
        try:
            return builder()
        except TypeError:
            for args in ((C.NUM_CLASSES, C.BEST_LR), (C.NUM_CLASSES,), ()):
                try:
                    return builder(*args)
                except TypeError:
                    continue
            raise

    for name, builder, dm, ckpt in C.VARIANTS[:len(C.B200_VARIANT_NAMES)]:     # the B200 variants; the rest are the reference's own
        lit = build_lit(builder)
        assert lit.hparams.num_classes == C.NUM_CLASSES and hasattr(lit, "training_step") and hasattr(lit, "configure_optimizers")
        assert hasattr(lit, "model") and isinstance(lit.model, torch.nn.Module)
        assert str(ckpt).endswith(name)
