"""CPU: pin the oracle restatement (oracle/spff_oracle.py) against outputs of the reference itself
(tests/golden/*.npz, written by oracle/make_golden.py from /root/reference). The reference ships no
tests or golden vectors of its own (SURVEY.md §4), so these fixtures are the pin.
Tolerances: both sides are CPU fp32 of the same operator sequence up to re-association (the oracle
evaluates gates functionally) -> logits 1e-4 abs / 1e-5 rel-L2, gradients 1e-3 rel on the norms."""
import glob
import os

import numpy as np
import pytest
import torch

from oracle import spff_oracle as O

GOLD = os.path.join(os.path.dirname(__file__), "golden")
CASES = sorted(glob.glob(os.path.join(GOLD, "case*.npz")))


def _load(path):
    z = np.load(path, allow_pickle=False)
    variant, b, h, w, ign, seed = [str(v) for v in z["case"]]
    return z, variant, int(b), int(h), int(w), float(ign), int(seed)


def test_fixtures_exist():
    assert len(CASES) >= 5 and os.path.exists(os.path.join(GOLD, "init_seed42.npz"))


@pytest.mark.usefixtures("reference_threads")
@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_oracle_matches_reference(path):
    z, variant, b, h, w, ign, seed = _load(path)
    x, lab = O.phantom_batch(b, h, w, seed=seed, ignore_frac=ign)
    p = O.det_weights(O.param_shapes(variant), seed=42)
    loss, logits, grads = O.loss_and_grads(p, x, lab, variant)
    ref = torch.from_numpy(z["logits"])
    assert logits.shape == ref.shape
    assert float((logits - ref).norm() / ref.norm()) < 1e-5
    assert float((logits - ref).abs().max()) < 1e-4
    assert abs(loss - float(z["loss"])) < 1e-5
    names = [str(n) for n in z["grad_names"]]
    assert sorted(names) == sorted(grads)
    for name, gn in zip(names, z["grad_norms"]):
        g = grads[name].double().reshape(-1)
        assert abs(float(g.norm()) - gn) <= 1e-3 * gn + 1e-7, name
        step = max(1, g.numel() // 512)
        sample = g[::step][:512].float().numpy()
        np.testing.assert_allclose(sample, z["g|" + name], rtol=2e-3, atol=2e-3 * (gn / max(1.0, g.numel() ** 0.5)) + 1e-7,
                                   err_msg=name)


@pytest.mark.parametrize("path", CASES, ids=[os.path.basename(p) for p in CASES])
def test_metrics_match_reference(path):
    z, variant, b, h, w, ign, seed = _load(path)
    _, lab = O.phantom_batch(b, h, w, seed=seed, ignore_frac=ign)
    logits = torch.from_numpy(z["logits"])
    m = O.per_class_metrics_3d(logits, lab, O.NUM_CLASSES, ignore_index=O.IGNORE_INDEX)
    np.testing.assert_allclose(np.array(m[0]), z["dice_list"], rtol=1e-12, equal_nan=True)
    np.testing.assert_allclose(np.array(m[1]), z["sens_list"], rtol=1e-12, equal_nan=True)
    np.testing.assert_allclose(np.array(m[2]), z["spec_list"], rtol=1e-12, equal_nan=True)
    np.testing.assert_allclose(np.array(m[3:]), z["scalars"], rtol=1e-12, equal_nan=True)
    lab0 = torch.where(lab == 255, torch.zeros_like(lab), lab)
    m2 = O.per_class_metrics_3d(logits, lab0, O.NUM_CLASSES)
    np.testing.assert_allclose(np.array(m2[3:]), z["scalars_noignore"], rtol=1e-12, equal_nan=True)
    # loss = CE + 0.5 * (1 - hard macro dice)
    loss = O.ce_plus_macro_dice_loss(logits, lab)
    assert abs(float(loss) - float(z["loss"])) < 1e-6


def test_parameter_surface_matches_reference():
    """state_dict keys / shapes of the oracle's parameter surface == the reference constructors'
    (plus the lazily registered freq_mask, models.py:1532-1535)."""
    z = np.load(os.path.join(GOLD, "init_seed42.npz"))
    by_variant = {}
    for key in z.files:
        variant, name = key.split("|")
        by_variant.setdefault(variant, {})[name] = tuple(int(v) for v in z[key][:-2])
    for variant, ref in by_variant.items():
        mine = {k: v for k, v in O.param_shapes(variant).items() if not k.endswith("freq_mask")}
        assert mine == ref, variant


def test_spff_tail_is_an_affine():
    """SURVEY.md §7.3: EFiLM -> FourierGate -> SpectralSE -> ChannelSE collapses to a*P + Q with P, Q
    functions of S_a = sum_hw a. Checked on the oracle's own gate functions."""
    torch.manual_seed(0)
    c, d = 32, 5
    shapes = {k: v for k, v in O.param_shapes("SPFF-UNet").items() if k.startswith("model.enc1.") or k.startswith("model.se.0")}
    p = O.det_weights(shapes, seed=3)
    a = torch.nn.functional.leaky_relu(torch.randn(2, c, d, 8, 8), 0.01)
    full = O._channel_se(p, "model.se.0", O._spectral_se(O._fgate(p, "model.enc1.fgate", O._efilm(p, "model.enc1.efilm", a))))
    g1, bt = O.efilm_tables(p, "model.enc1.efilm", c, d)
    hw = 64
    S = a.sum(dim=(3, 4))                                   # [B,C,D]
    Se = S * g1 + bt * hw
    s = Se.sum(1) / (c * hw)                                 # [B,D]
    m = (p["model.enc1.fgate.freq_mask"] * p["model.enc1.fgate.mag_scale"]).reshape(-1)
    w1 = torch.sigmoid(torch.fft.irfft(torch.fft.rfft(s, dim=1) * m, n=d, dim=1))
    Sf = Se * w1[:, None, :]
    w2 = torch.sigmoid(Sf.sum(1) / (c * hw))
    Sg = Sf * w2[:, None, :]
    z = Sg.sum(2) / (d * hw)                                 # [B,C]
    W1 = p["model.se.0.fc.0.weight"].reshape(-1, c); W2 = p["model.se.0.fc.2.weight"].reshape(c, -1)
    w3 = torch.sigmoid(torch.relu(z @ W1.t() + p["model.se.0.fc.0.bias"]) @ W2.t() + p["model.se.0.fc.2.bias"])
    P = g1[None] * w1[:, None, :] * w2[:, None, :] * w3[:, :, None]
    Q = bt[None] * w1[:, None, :] * w2[:, None, :] * w3[:, :, None]
    aff = a * P[..., None, None] + Q[..., None, None]
    assert float((aff - full).abs().max()) < 1e-5
