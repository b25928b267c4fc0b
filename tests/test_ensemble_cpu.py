"""CPU half of the ensemble / mirror-TTA path: SpctEnsemble's refusals of members it cannot average, the flip tables
that turn spff_grid_aug into torch.flip, and the sample-group sizing with the ensemble's extra per-sample footprint."""
import pytest
import torch


def _variant(name, seed=0, **kw):
    from innovative3D import config as C
    torch.manual_seed(seed)
    return dict((v[0], v[1]) for v in C.VARIANTS)[name](**kw)


def test_ensemble_accepts_spct_members_and_cores():
    from innovative3D import models
    a, b = _variant("SPFF-UNet", 1), _variant("SPFF-UNet", 2)
    ens = models.SpctEnsemble([a, b.model], tta="flip")
    assert ens.cores == [a.model, b.model] and ens.flips == (0, 1, 2, 3) and ens.num_classes == 13
    assert ens.cores[0] is a.model                     # references, no copies of the weights
    assert models.SpctEnsemble([_variant("PlainCore_UNet")]).flips == (0,)
    for name in ("E_SP_UNet", "FG_SP_UNet"):
        models.SpctEnsemble([_variant(name, 1), _variant(name, 2)])


def test_ensemble_refusals():
    from innovative3D import models
    spff = _variant("SPFF-UNet")
    with pytest.raises(ValueError, match="at least one member"):
        models.SpctEnsemble([])
    for bad in ("rot90", "FLIP", 1):
        with pytest.raises(ValueError, match="tta"):
            models.SpctEnsemble([spff], tta=bad)
    with pytest.raises(NotImplementedError, match="SP_UNet"):
        models.SpctEnsemble([spff, _variant("SP_UNet")])
    cicek = models.LitCicek3DUNet_DepthAdapter_Published(num_classes=13)
    with pytest.raises(NotImplementedError, match="BatchNorm"):
        models.SpctEnsemble([spff, cicek])
    with pytest.raises(NotImplementedError, match="BatchNorm"):
        models.SpctEnsemble([cicek.backbone])
    with pytest.raises(ValueError, match="'efilm'"):          # SPFF-UNet vs FG_SP_UNet: EnergyFiLM differs
        models.SpctEnsemble([spff, _variant("FG_SP_UNet")])
    with pytest.raises(ValueError, match="'fgate'"):
        models.SpctEnsemble([spff, _variant("E_SP_UNet")])
    with pytest.raises(ValueError, match="'num_classes'"):
        models.SpctEnsemble([spff, models.LitSPCT_EFiLM_FourierGate(num_classes=5)])
    with pytest.raises(TypeError):
        models.SpctEnsemble([spff, torch.nn.Linear(2, 2)])


def test_ensemble_construction_touches_no_member_state():
    from innovative3D import models
    a = _variant("SPFF-UNet", 4)
    before = {k: v.clone() for k, v in a.state_dict().items()}
    models.SpctEnsemble([a, a], tta="flip")
    assert a._fused is None and a._copy_stream is None
    assert all(torch.equal(before[k], v) for k, v in a.state_dict().items())


@pytest.mark.parametrize("flip", [1, 2, 3])
def test_flip_tables_are_torch_flip(flip):
    """spff_grid_aug gathers xo[n][f][u][v] = x[n][f][amap[n][u]][bmap[n][v]] (no transpose, no jitter): with these
    tables that is torch.flip over the flipped axes."""
    from spff_b200.engine import flip_tables
    n, f, h, w = 3, 5, 8, 16
    x = torch.randn(n, f, h, w, generator=torch.Generator().manual_seed(flip))
    amap, bmap = flip_tables(n, h, w, flip)
    assert amap.dtype == torch.int32 and tuple(amap.shape) == (n, h) and tuple(bmap.shape) == (n, w)
    gathered = torch.stack([x[i][:, amap[i].long()][:, :, bmap[i].long()] for i in range(n)])
    dims = [d for bit, d in ((1, 2), (2, 3)) if flip & bit]
    assert torch.equal(gathered, torch.flip(x, dims))


def test_sample_group_sizing_with_extra_footprint(monkeypatch):
    """fit_group's default keeps today's units; the ensemble adds its fp32 accumulator (64 B per position: one level-1
    unit) and the fp32 flipped input (4 B: 1/16 unit) per sample."""
    from spff_b200.engine import ENSEMBLE_UNITS, SpffEngine
    free = 170 * 2 ** 30
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (free, 183 * 2 ** 30))
    unit = 5 * 512 * 512 * 64
    assert ENSEMBLE_UNITS == 1.0 + 4 / 64
    assert SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=False) == int(0.45 * free / (16.7 * unit)) == 58
    assert SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=False, extra=0.0) == 58
    got = SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=False, extra=ENSEMBLE_UNITS)
    assert got == int(0.45 * free / ((16.7 + ENSEMBLE_UNITS) * unit)) == 55
    assert SpffEngine.fit_group(256, 5, 128, 128, "cuda:0", train=False, extra=ENSEMBLE_UNITS) == 256
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda device=None: (2 ** 30, 183 * 2 ** 30))
    assert SpffEngine.fit_group(256, 5, 512, 512, "cuda:0", train=False, extra=ENSEMBLE_UNITS) == 1
