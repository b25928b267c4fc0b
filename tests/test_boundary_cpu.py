"""The plugin boundary (SURVEY.md §8b), no GPU needed: with a reference checkout's `innovative3D/` directory on the
package path, this tree's `innovative3D` keeps the hot-path names and hands every other name through to the reference's
module of the same name (`_fallthrough.py`). The checkout here is a minimal stand-in written to a temporary directory
with the layout of the reference's (a namespace directory without `__init__.py`, holding `config.py`, `helpers.py`,
`models.py` and `datasets.py`), so the test needs nothing outside this repository.
Covers the name collision of round 1 (`innovative3D.datasets` of this tree shadowing the reference's data layer)."""
import json
import os
import subprocess
import sys
import textwrap

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "spff-unet-spcct_b200")

B200 = ["SPFF-UNet", "E_SP_UNet", "FG_SP_UNet", "SP_UNet", "PlainCore_UNet", "3DUNet"]
OTHER_FAMILIES = ["UNETR", "SwinUNETR", "R2UNet", "ResUNet++"]

REFERENCE_FILES = {
    "config.py": f"""
        trainval_sets = [{{"name": f"scan{{i}}", "original_rois": [], "frames": 5}} for i in range(4)]
        test_set = [{{"name": "scan4", "original_rois": [], "frames": 5}}]

        def _builder():
            return None

        # the reference registers the B200 variants first, then the four other families (config.py:316-391)
        VARIANTS = [(name, _builder, None, "runs/" + name) for name in {B200 + OTHER_FAMILIES!r}]
    """,
    "helpers.py": """
        def create_image_and_labels_for_dataset(config):
            return config

        def generate_cumulative_grid_sizes(sizes):
            return sizes
    """,
    "models.py": """
        class R2UNet3D:
            pass

        class LitSPCT_ControlUNet:      # same name as this tree's class: must never win over it
            pass
    """,
    "datasets.py": """
        class DicomDataset3D:
            pass

        class MultiDicomDataModule3D:
            def __init__(self, configs, batch_size=1, num_frames=5):
                self.configs, self.batch_size, self.num_frames = configs, batch_size, num_frames
    """,
}


@pytest.fixture(scope="module")
def reference_checkout(tmp_path_factory):
    """A reference-shaped `innovative3D/` portion appended to this package's __path__, removed afterwards."""
    for p in (ROOT, PKG):
        if p not in sys.path:
            sys.path.insert(0, p)
    import innovative3D
    ref = tmp_path_factory.mktemp("reference") / "innovative3D"
    ref.mkdir()
    for name, body in REFERENCE_FILES.items():
        (ref / name).write_text(textwrap.dedent(body))
    innovative3D.__path__.append(str(ref))
    yield ref
    innovative3D.__path__.remove(str(ref))
    for k in [k for k in sys.modules if k == "innovative3D.datasets" or k.startswith("innovative3D._reference_")]:
        del sys.modules[k]


def test_package_shadows_hot_path_and_falls_through_for_the_rest(reference_checkout):
    import innovative3D
    import innovative3D.config as C
    import innovative3D.helpers as H
    import innovative3D.models as M
    here = PKG
    assert innovative3D.__file__.startswith(here) and C.__file__.startswith(here) and M.__file__.startswith(here)
    # hot-path names are this tree's
    assert M.LitSPCT_EFiLM_FourierGate.__module__ == "innovative3D.models"
    assert H.ce_plus_macro_dice_loss.__module__ == "innovative3D.helpers"
    # the data layer is the reference's: its module, its tables, its ingest helpers
    import innovative3D.datasets as D
    assert D.__file__.startswith(str(reference_checkout)) and hasattr(D, "MultiDicomDataModule3D") and hasattr(D, "DicomDataset3D")
    assert len(C.trainval_sets) == 4 and len(C.test_set) == 1 and "original_rois" in C.trainval_sets[0]
    dm = C.MultiDicomDataModule3D(C.trainval_sets, batch_size=1, num_frames=C.NUM_FRAMES)      # as train.py:1410 builds it
    assert type(dm) is D.MultiDicomDataModule3D and dm.batch_size == 1 and len(dm.configs) == 4
    assert callable(H.create_image_and_labels_for_dataset) and callable(H.generate_cumulative_grid_sizes)
    assert H.create_image_and_labels_for_dataset.__module__ == "innovative3D._reference_helpers"
    with pytest.raises(AttributeError, match="B200 hot-path build"):
        C.no_such_name
    # this tree's GPU data path lives under its own name
    from innovative3D.datapath_gpu import TrainGridAug   # noqa: F401


def test_other_families_resolve_to_the_reference_code(reference_checkout):
    import innovative3D.models as M
    cls = M.R2UNet3D if hasattr(M, "R2UNet3D") else None
    ref_models = sys.modules.get("innovative3D._reference_models")
    assert ref_models is not None, "models.py fall-through did not load the reference module"
    assert cls is not None and cls.__module__ == "innovative3D._reference_models"
    assert M.LitSPCT_ControlUNet.__module__ == "innovative3D.models"      # never the reference's class of the same name


def test_reference_variants_are_appended_after_the_b200_ones(reference_checkout):
    """`config._append_reference_variants` runs when `innovative3D.config` is first imported: a fresh interpreter with
    the checkout on sys.path keeps the B200 entries and appends the reference's other families, its own objects."""
    code = textwrap.dedent("""
        import json, sys
        sys.path[:0] = sys.argv[1:3]
        sys.path.append(sys.argv[3])
        import innovative3D.config as C
        print(json.dumps([[v[0], v[1].__module__] for v in C.VARIANTS]))
    """)
    out = subprocess.run([sys.executable, "-c", code, ROOT, PKG, str(reference_checkout.parent)],
                         capture_output=True, text=True, check=True)
    variants = json.loads(out.stdout.strip().splitlines()[-1])
    assert [n for n, _ in variants] == B200 + OTHER_FAMILIES
    assert all(m == "innovative3D.config" for _, m in variants[:6])
    assert all(m == "innovative3D._reference_config" for _, m in variants[6:])


def test_cpu_forward_is_loud_not_a_fallback():
    import torch

    from innovative3D import config as C
    lit = dict((v[0], v[1]) for v in C.VARIANTS)["SPFF-UNet"]()
    with pytest.raises(RuntimeError, match="no CPU"):
        lit(torch.zeros(1, 1, 5, 16, 16))
