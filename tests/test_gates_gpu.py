"""GPU: the SPFF gate kernels of csrc/gates.cu against an fp64 reference built from the oracle's gate definitions.

The four entry points, called through `spff_b200.ops`:
- `gate_tables_fwd` / `gate_tables_bwd`: the parameter-only tables g1, bt [c, frames] (EnergyFiLM's MLP over the
  sinusoidal bin code) and kfg [frames] (FourierGate's irfft(freq_mask * mag_scale)), and the parameter gradients
  folded back from the table gradients;
- `gate_micro_fwd` / `gate_micro_bwd`: the plane sums S [n, d, c] -> out = a * P + Q, and the InstanceNorm backward
  coefficients, dS, P and every gate-parameter gradient from the backward plane sums R [n, d, c, 6].

The reference is the oracle's EnergyFiLM -> FourierGate -> SpectralSE -> ChannelSE chain in fp64 with autograd for the
gradients (`efilm_tables`, `_efilm`, `_fgate`, `_spectral_se`, `_channel_se`; irfft in complex128), in two tiers:
- full tensors: a = lrelu(IN(x)), out = tail(a), L = sum dout * out on small planes; with g1, bt, kfg as leaf tensors
  autograd gives the table gradients the micro kernel produces;
- plane sums: every gate sees the activation only through plane means, so the tail of the two-pixel plane
  {m + 1, m - 1}, m = S / hw, is exactly (m +- 1) P + Q. That gives P and Q as functions of S, and
  L = sum P * R[0] + Q * R[1] (R[0] = sum dout * a, R[1] = sum dout) their gradients, at any plane size up to
  512 x 512 without the tensors. `test_reference_tiers_agree` shows the two tiers equal to fp64 precision first.
The kernel inputs (S, R, coef, tables, weights) are rounded once to fp32 and the reference takes those rounded values,
so a comparison measures the kernel's own error only.

Tolerances. The kernels compute in fp32 and store nothing narrower. Their error sources:
- fp32 sums inside a CTA: over c (a per-thread stride-256 loop of <= 2 terms, a 5-level warp tree, 8 warp partials
  in sequence), over d <= 16, over hid <= 64, and in the table kernels over 2c <= 1024 terms in sequence;
- fp32 atomics across the n <= 37 samples of a call (dgamma, dbeta, dg1, dbt, dkfg, dse_*), in any order;
- `__expf` in the sigmoids: x * log2(e) rounded once, so a relative error of about |x| u plus the 2 ulp of ex2.approx;
  the sigmoid arguments here stay below ~10 in magnitude, so below 1e-6.
A sum of N random-sign terms errs by about u sqrt(N) of its result (each partial sum is rounded, and the terms add up
to sqrt(N) times the result: Higham & Mary, SIAM J. Sci. Comput. 41(5), 2019), and sums in sequence multiply these
factors. Each output is compared on its largest entry: max |kernel - reference| <= tol * max |reference|, with
- TOL = 2e-5 for everything computed per sample (P, Q, Pout, dSa, bcoef.y, bcoef.z) and for the table kernels, whose
  sums run in a fixed order. The longest chain is the 2c = 1024-term sum of the table backward, u sqrt(1024) = 2e-6;
  the largest seen on a B200 is a quarter of the bound (dmag_scale);
- TOL_ACC = 5e-5 for the gradients the micro kernel accumulates over samples with atomics: a c-sum, a d-sum and the
  n-sum in sequence, u sqrt(512 * 16 * 37) = 3.3e-5 at the largest case. The atomics' order changes from run to run;
  the largest seen is 1.3e-5 (dkfg at d = 1, c = 512, n = 37, where each sample's term is itself a 512-channel sum).
Both are at least 100x tighter than the 5e-3 of the end-to-end tail tests, whose bound comes from the bf16
activations in front of these kernels. Exceptions, each exact: bcoef.x = fp32(gamma * rstd) is one rounding
(u relative), bcoef.w and every Q of a block without EnergyFiLM are 0, and the outputs a call does not own keep their
NaN fill. Outputs that accumulate (+=) start from random contents of the gradient's own magnitude, which adds one
rounding, 2u of the result, to each bound.
"""
import contextlib
import math
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U = 2.0 ** -24          # fp32 unit roundoff
TOL = 2e-5              # per-sample outputs and the table kernels: see the module docstring
TOL_ACC = 5e-5          # gradients the micro kernel accumulates over samples with atomics
SLOPE, EPS = 0.01, 1e-5
EFILM, FOURIER, SPECSE, CHANSE = 1, 2, 4, 8      # SPFF_GATE_* of include/spff_b200.h
WORST = {}              # output -> (worst error / bound seen, test that saw it)
CURRENT = [""]          # the running test's id


# --------------------------------------------------------------------------------------------------------------------
# fp64 reference
# --------------------------------------------------------------------------------------------------------------------
def pe64(frames, d):
    """oracle.sinusoidal_pe, in fp64 (the oracle builds the code in fp32)."""
    pos = torch.arange(frames, dtype=torch.float64)[None, None, :]
    i = torch.arange(max(1, d // 2), dtype=torch.float64)[None, :, None]
    denom = torch.exp(i * (-math.log(10000.0) / max(1, d // 2)))
    pe = torch.cat([torch.sin(pos * denom), torch.cos(pos * denom)], dim=1)
    if pe.shape[1] < d:
        pe = torch.cat([pe, torch.zeros(1, 1, pe.shape[-1], dtype=torch.float64)], dim=1)
    return pe


@contextlib.contextmanager
def fp64_oracle():
    """The oracle's EnergyFiLM with an fp64 positional code."""
    from oracle import spff_oracle as O
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(O, "sinusoidal_pe", pe64)
        yield O


def ref_tables(p, c, frames, efilm=True, fgate=True):
    """g1, bt [c, frames] (oracle.efilm_tables) and kfg [frames] = irfft(freq_mask * mag_scale) of the fp64 parameters
    p["e.mlp.*"], p["f.*"]; None for a gate left out."""
    g1 = bt = kfg = None
    if efilm:
        with fp64_oracle() as O:
            g1, bt = O.efilm_tables(p, "e", c, frames)
    if fgate:
        spec = (p["f.freq_mask"] * p["f.mag_scale"]).reshape(-1).to(torch.complex128)
        kfg = torch.fft.irfft(spec, n=frames)
    return g1, bt, kfg


def tail64(x, flags, g1=None, bt=None, kfg=None, se=None):
    """The gate chain of a block (oracle.core_forward: EFiLM -> FourierGate -> SpectralSE -> ChannelSE) on
    x [n, c, d, h, w] with the parameter-only tables as inputs. EFiLM applies g1, bt as oracle._efilm does;
    FourierGate is oracle._fgate with its spectrum freq_mask * mag_scale written as rfft(kfg), which is the same
    thing when kfg = irfft(freq_mask * mag_scale), and for any other real kfg a circular convolution with it.
    se: oracle._channel_se's parameters under the prefix "s"."""
    from oracle import spff_oracle as O
    if flags & EFILM:
        x = x * g1[None, :, :, None, None] + bt[None, :, :, None, None]
    if flags & FOURIER:
        s = x.mean(dim=(1, 3, 4), keepdim=True)
        w = torch.fft.irfft(torch.fft.rfft(s, dim=2) * torch.fft.rfft(kfg)[None, None, :, None, None], n=x.shape[2], dim=2)
        x = x * torch.sigmoid(w)
    if flags & SPECSE:
        x = O._spectral_se(x)
    if flags & CHANSE:
        x = O._channel_se(se, "s", x)
    return x


def plane_pq(S, hw, tail):
    """P, Q [n, d, c] of out = a * P + Q from the plane sums S [n, d, c] of planes of hw positions: the tail of the
    two-pixel plane {m + 1, m - 1}, m = S / hw, whose mean is that of the real plane."""
    m = (S / hw).permute(0, 2, 1)[..., None, None]                      # [n, c, d, 1, 1]
    o = tail(torch.cat([m + 1, m - 1], dim=4))
    P = (o[..., 0] - o[..., 1]) / 2
    Q = (o[..., 0] + o[..., 1]) / 2 - m[..., 0] * P
    return P[..., 0].permute(0, 2, 1), Q[..., 0].permute(0, 2, 1)


def plane_reference(S, R, hw, tail, leaves):
    """Everything gate_micro_fwd / _bwd compute, from the plane sums S [n, d, c] and R [n, d, c, 6] =
    sums over (h, w) of {dout*a, dout, dout*m, m, dout*m*xhat, m*xhat} (m = lrelu'): P, Q, dSa = dL/dS, the
    per-(n, c) sums of dz = dL/d(IN output) and dz * xhat, and dL/d(leaf) for every leaf (None where unused)."""
    S = S.detach().clone().requires_grad_()
    P, Q = plane_pq(S, hw, tail)
    L = (P * R[..., 0] + Q * R[..., 1]).sum()
    g = torch.autograd.grad(L, [S] + list(leaves), allow_unused=True)
    dSa = g[0] if g[0] is not None else torch.zeros_like(S)
    P = P.detach()
    return dict(P=P, Q=Q.detach(), dSa=dSa,
                sum_dz=(P * R[..., 2] + dSa * R[..., 3]).sum(1), sum_dzx=(P * R[..., 4] + dSa * R[..., 5]).sum(1),
                grads=g[1:])


def instance_stats(x):
    """rstd [n, c, 1, 1, 1] and xhat of InstanceNorm3d(eps 1e-5) on x [n, c, d, h, w]."""
    mean = x.mean(dim=(2, 3, 4), keepdim=True)
    rstd = (x.var(dim=(2, 3, 4), unbiased=False, keepdim=True) + EPS).rsqrt()
    return rstd, (x - mean) * rstd


def se_dict(w1, b1, w2, b2):
    hid, c = w1.shape
    return {"s.fc.0.weight": w1.reshape(hid, c, 1, 1, 1), "s.fc.0.bias": b1,
            "s.fc.2.weight": w2.reshape(c, hid, 1, 1, 1), "s.fc.2.bias": b2}


# --------------------------------------------------------------------------------------------------------------------
# inputs and checks
# --------------------------------------------------------------------------------------------------------------------
def q32(t):
    """Round to fp32 once; the kernel takes the fp32 value and the reference the same value in fp64."""
    return t.float().double()


def gen(seed):
    g = torch.Generator().manual_seed(seed)
    return lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)


def plane_inputs(r, n, c, d, hw):
    """S, R with the magnitudes of an IN + LeakyReLU output and its gradient over hw positions (means of a near 0.4,
    of m near 0.5, gradient sums growing like sqrt(hw)), coef {A, B, mean, rstd} and gamma with a zero and a negative
    entry."""
    sq = math.sqrt(hw)
    S = q32(hw * (0.4 + 0.3 * r(n, d, c)))
    R = q32(torch.stack([0.6 * sq * r(n, d, c), sq * r(n, d, c), 0.7 * sq * r(n, d, c), hw * (0.5 + 0.1 * r(n, d, c)),
                         0.6 * sq * r(n, d, c), hw * (0.4 + 0.1 * r(n, d, c))], dim=-1))
    gamma = q32(1 + 0.3 * r(c))
    gamma[0], gamma[1] = 0.0, -0.7
    rstd, mean, beta = torch.exp(0.5 * r(n, c)), r(n, c), 0.1 * r(c)
    A = rstd * gamma
    coef = q32(torch.stack([A, beta - mean * A, mean, rstd], dim=-1))
    return S, R, coef, gamma


def micro_params(r, c, d, hid):
    """Tables and SE weights at the scale of the trained ones (det_weights' fan-in scaling). kfg is a general real
    kernel, not only a symmetric one like irfft(freq_mask * mag_scale), so that the convolution's direction
    (kfg[t - e] rather than kfg[e - t]) is checked in the forward and in dkfg."""
    return dict(g1=q32(1 + torch.tanh(0.5 * r(c, d))), bt=q32(0.2 * r(c, d)), kfg=q32(0.5 * r(d)),
                w1=q32(r(hid, c) * 1.5 / math.sqrt(c)), b1=q32(0.1 * r(hid)), w2=q32(r(c, hid) * 1.5 / math.sqrt(hid)),
                b2=q32(0.1 * r(c)))


def cu(t):
    return t.float().contiguous().cuda()


def nan(*shape):
    return torch.full(shape, float("nan"), device="cuda")


def check(name, got, want, tol=TOL, init=None, floor=0.0):
    """max |got - want| <= tol * max |want| + floor (+ 2u of the result when got accumulated onto `init`)."""
    got, want = got.double().cpu(), want.double().cpu()
    assert got.shape == want.shape, (name, tuple(got.shape), tuple(want.shape))
    bound = tol * float(want.abs().max()) + floor
    if init is not None:
        want = want + init.double().cpu()
        bound += 2 * U * float(want.abs().max())
    err = float((got - want).abs().max())
    key = name.split("[")[0]
    WORST[key] = max(WORST.get(key, (0.0, "")), (err / bound if bound > 0 else float(err > 0), CURRENT[0]))
    assert err <= bound, f"{name}: max error {err:.3e} > bound {bound:.3e} (max |reference| {float(want.abs().max()):.3e})"


def dsa_floor(R, hw):
    """The reference's own rounding in dS: P and Q come from differences of O(1) values in fp64, and dS from
    L = sum P R[0] + Q R[1] with m = S / hw, so its noise is about 1e-16 (|R[0]| + |R[1]|) / hw. Where dS is 0 (a block
    with EnergyFiLM alone, whose P and Q do not depend on S, or a ChannelSE with every hidden unit cut by the ReLU)
    the kernel writes exact zeros against that noise; a wrong term of any size shows far above 1e-12 of the scale."""
    return 1e-12 * float((R[..., 0].abs() + R[..., 1].abs()).max()) / hw


def untouched(name, t):
    assert torch.isnan(t).all(), f"{name}: written although the call does not own it"


@pytest.fixture(autouse=True)
def _budget(request):
    """Per-test runtime and peak allocation (the machines are shared: every test frees what it allocated)."""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    CURRENT[0] = request.node.name
    yield
    torch.cuda.synchronize()
    print(f"\n[budget] {request.node.name}: {time.time() - t0:.2f} s, peak {torch.cuda.max_memory_allocated() / 2 ** 30:.3f} GiB")
    torch.cuda.empty_cache()


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / bound per output:")
        for k in sorted(WORST):
            print(f"  {k:16s} {WORST[k][0]:.3f}  {WORST[k][1]}")


# --------------------------------------------------------------------------------------------------------------------
# 0. the two reference tiers agree
# --------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("flags", range(16))
@pytest.mark.parametrize("n,c,d,h,w,hid", [(2, 8, 5, 3, 4, 3), (1, 12, 4, 5, 2, 1), (2, 16, 16, 2, 3, 4)])
def test_reference_tiers_agree(flags, n, c, d, h, w, hid):
    """On small planes, in fp64: (1) the tail with table leaves equals the oracle's own EFiLM / FourierGate built from
    the MLP and mask parameters, output and parameter gradients; (2) the plane-sum tier gives out = a * P + Q and the
    full tensor's autograd gradients: dS through the InstanceNorm backward dx = gamma rstd (dz - mean dz -
    xhat mean(dz xhat)), dz = (dout P + dS) m, and dgamma, dbeta, dg1, dbt, dkfg and the SE weight gradients."""
    r = gen(100 + flags)
    x = (1.3 * r(n, c, d, h, w) + 0.3).requires_grad_()
    dout = r(n, c, d, h, w)
    gamma = (1 + 0.3 * r(c)).requires_grad_()
    beta = (0.2 * r(c)).requires_grad_()
    p = {"e.mlp.0.weight": 0.3 * r(32, 16, 1), "e.mlp.0.bias": 0.1 * r(32), "e.mlp.2.weight": 0.3 * r(2 * c, 32, 1),
         "e.mlp.2.bias": 0.1 * r(2 * c), "f.freq_mask": 1 + 0.2 * r(1, 1, d // 2 + 1, 1, 1), "f.mag_scale": 1 + 0.1 * r(1)}
    for v in p.values():
        v.requires_grad_()
    sw = [(0.4 * r(hid, c)).requires_grad_(), (0.1 * r(hid)).requires_grad_(), (0.4 * r(c, hid)).requires_grad_(),
          (0.1 * r(c)).requires_grad_()]
    se = se_dict(*sw)
    z = F.instance_norm(x, weight=gamma, bias=beta, eps=EPS)
    a = F.leaky_relu(z, SLOPE)

    # (1) oracle route, from the parameters
    from oracle import spff_oracle as O
    with fp64_oracle():
        o = a
        if flags & EFILM:
            o = O._efilm(p, "e", o)
        if flags & FOURIER:
            o = O._fgate(p, "f", o)
    out_oracle = tail64(o, flags & (SPECSE | CHANSE), se=se)
    params = list(p.values())
    g_oracle = torch.autograd.grad((dout * out_oracle).sum(), params, retain_graph=True, allow_unused=True)

    # table leaves
    g1p, btp, kfgp = ref_tables(p, c, d)
    g1, bt, kfg = (t.detach().clone().requires_grad_() for t in (g1p, btp, kfgp))
    out = tail64(a, flags, g1, bt, kfg, se)
    torch.testing.assert_close(out, out_oracle, rtol=1e-12, atol=1e-12)
    L = (dout * out).sum()
    leaves = [g1, bt, kfg] + sw
    full = torch.autograd.grad(L, [x, gamma, beta, z] + leaves, allow_unused=True)
    g_tables = torch.autograd.grad([g1p, btp, kfgp], params,
                                   [t if t is not None else torch.zeros_like(l) for t, l in zip(full[4:7], (g1, bt, kfg))],
                                   allow_unused=True)
    for name, ga, gb in zip(p, g_oracle, g_tables):
        if ga is not None:
            torch.testing.assert_close(gb, ga, rtol=1e-10, atol=1e-12, msg=name)

    # (2) plane-sum tier from the full tensor's sums
    rstd, xhat = instance_stats(x.detach())
    zd, ad = z.detach(), a.detach()
    mslope = torch.where(zd > 0, torch.ones_like(zd), torch.full_like(zd, SLOPE))
    hw = h * w
    pl = lambda t: t.sum(dim=(3, 4)).permute(0, 2, 1)       # [n, c, d, h, w] -> plane sums [n, d, c]
    S = pl(ad)
    R = torch.stack([pl(dout * ad), pl(dout), pl(dout * mslope), pl(mslope), pl(dout * mslope * xhat), pl(mslope * xhat)], -1)
    ref = plane_reference(S, R, hw, lambda t: tail64(t, flags, g1, bt, kfg, se), leaves)
    P5 = ref["P"].permute(0, 2, 1)[..., None, None]
    Q5 = ref["Q"].permute(0, 2, 1)[..., None, None]
    torch.testing.assert_close(ad * P5 + Q5, out.detach(), rtol=1e-11, atol=1e-11)
    dz = (dout * P5 + ref["dSa"].permute(0, 2, 1)[..., None, None]) * mslope
    torch.testing.assert_close(dz, full[3], rtol=1e-10, atol=1e-11)
    cnt = d * hw
    c1 = (gamma.detach() * rstd[:, :, 0, 0, 0])[..., None, None, None]
    c2 = (ref["sum_dz"] / cnt)[..., None, None, None]
    c3 = (ref["sum_dzx"] / cnt)[..., None, None, None]
    torch.testing.assert_close(c1 * (dz - c2 - xhat * c3), full[0], rtol=1e-10, atol=1e-11)
    torch.testing.assert_close(ref["sum_dzx"].sum(0), full[1], rtol=1e-10, atol=1e-11)
    torch.testing.assert_close(ref["sum_dz"].sum(0), full[2], rtol=1e-10, atol=1e-11)
    for name, gp, gf in zip(("dg1", "dbt", "dkfg", "dse_w1", "dse_b1", "dse_w2", "dse_b2"), ref["grads"], full[4:]):
        if gf is None:
            assert gp is None or not gp.abs().max() > 1e-14, name
        else:
            torch.testing.assert_close(gp, gf, rtol=1e-10, atol=1e-11, msg=name)


# --------------------------------------------------------------------------------------------------------------------
# 1, 2. the table kernels
# --------------------------------------------------------------------------------------------------------------------
TABLE_C = (32, 64, 128, 256, 512)
GATE_SETS = {"efilm": (True, False), "fourier": (False, True), "both": (True, True), "neither": (False, False)}


def table_params(r, c, frames):
    """fp32-exact fp64 parameters of one block's EFiLM MLP and FourierGate mask (det_weights' scales)."""
    return {"e.mlp.0.weight": q32(0.3 * r(32, 16, 1)), "e.mlp.0.bias": q32(0.1 * r(32)),
            "e.mlp.2.weight": q32(0.27 * r(2 * c, 32, 1)), "e.mlp.2.bias": q32(0.1 * r(2 * c)),
            "f.freq_mask": q32(1 + 0.2 * r(1, 1, frames // 2 + 1, 1, 1)), "f.mag_scale": q32(1 + 0.1 * r(1))}


def table_args(p, efilm, fgate):
    e = [cu(p[k]) for k in ("e.mlp.0.weight", "e.mlp.0.bias", "e.mlp.2.weight", "e.mlp.2.bias")] if efilm else [None] * 4
    f = [cu(p["f.freq_mask"].reshape(-1)), cu(p["f.mag_scale"])] if fgate else [None] * 2
    return e + f


@pytest.mark.parametrize("gates", list(GATE_SETS))
@pytest.mark.parametrize("frames", range(1, 17))
def test_gate_tables_fwd(frames, gates):
    """g1, bt, kfg for every bin count (odd and even F weight the Nyquist bin differently) and channel count; a gate
    left out writes nothing."""
    from spff_b200 import ops
    efilm, fgate = GATE_SETS[gates]
    for c in TABLE_C:
        p = table_params(gen(1000 * frames + c), c, frames)
        g1, bt, kfg = nan(c, frames), nan(c, frames), nan(frames)
        ops.gate_tables_fwd(*table_args(p, efilm, fgate), c, frames, g1, bt, kfg)
        torch.cuda.synchronize()
        rg1, rbt, rkfg = ref_tables(p, c, frames)
        for name, got, want, on in (("g1", g1, rg1, efilm), ("bt", bt, rbt, efilm), ("kfg", kfg, rkfg, fgate)):
            if on:
                check(f"{name}[c={c},F={frames}]", got, want)
            else:
                untouched(f"{name}[c={c},F={frames}]", got)


TABLE_BWD = [(f, c, "both") for f in range(1, 17) for c in (32, 512)] + \
            [(f, 256, g) for f in (4, 5, 16) for g in ("efilm", "fourier")]


@pytest.mark.parametrize("frames,c,gates", TABLE_BWD, ids=[f"F{f}-c{c}-{g}" for f, c, g in TABLE_BWD])
def test_gate_tables_bwd(frames, c, gates):
    """dw0, db0, dw2, db2, dfreq_mask, dmag_scale += autograd of sum dg1 g1 + dbt bt + dkfg kfg. c = 512 with F = 16
    needs 69 KB of dynamic shared memory, past the 48 KB default."""
    from spff_b200 import ops
    efilm, fgate = GATE_SETS[gates]
    r = gen(7000 + 31 * frames + c)
    p = table_params(r, c, frames)
    dg1, dbt, dkfg = q32(r(c, frames)), q32(r(c, frames)), q32(r(frames))
    leaves = {k: v.clone().requires_grad_() for k, v in p.items()}
    g1, bt, kfg = ref_tables(leaves, c, frames)
    L = (dg1 * g1).sum() + (dbt * bt).sum() + (dkfg * kfg).sum()
    keys = [k for k in p if (efilm and k.startswith("e.")) or (fgate and k.startswith("f."))]
    grads = dict(zip(keys, torch.autograd.grad(L, [leaves[k] for k in keys])))
    names = ("e.mlp.0.weight", "e.mlp.0.bias", "e.mlp.2.weight", "e.mlp.2.bias", "f.freq_mask", "f.mag_scale")
    # accumulators start from random contents of the gradient's magnitude (the kernel adds)
    init = {k: q32(r(*p[k].shape) * float(grads[k].abs().max() if k in grads else 1.0)) for k in names}
    out = {k: cu(init[k]) if k in grads else nan(*p[k].shape) for k in names}
    ops.gate_tables_bwd(*table_args(p, efilm, fgate), c, frames, cu(dg1), cu(dbt), cu(dkfg),
                        *(out[k] if k in grads else None for k in names))
    torch.cuda.synchronize()
    for k in names:
        if k in grads:
            check(f"d{k}[c={c},F={frames}]", out[k], grads[k], init=init[k])
        else:
            untouched(k, out[k])


# --------------------------------------------------------------------------------------------------------------------
# 3, 4. the micro kernels
# --------------------------------------------------------------------------------------------------------------------
DS = (1, 3, 5, 8, 9, 15, 16)            # <8,0> for d <= 8, <5,5> for d == 5, <16,0> up to 16: each and its edges
CS = (32, 64, 128, 256, 512)            # 256: one channel per thread; 512: two
NS = (1, 3, 37)                         # one CTA per sample
HWS = ((1, 1), (4, 4), (25, 17), (64, 64), (200, 136), (512, 512))


def _micro_grid():
    """Every flag combination at every d; c, n and the plane size rotate so that each flag set meets every c and n,
    and each d every c, n and plane size. Then the SE hidden width's limits (1 and kMaxHid = 64), and the encoder
    flags of SP_UNet (12), E_SP_UNet (13) and FG_SP_UNet (14) at d = 16, c = 256."""
    out = []
    for f in range(16):
        for j, d in enumerate(DS):
            i = 7 * f + j
            c = CS[i % 5]
            out.append((f, d, c, max(4, c // 16), NS[i % 3], HWS[i % 6]))
    out += [(15, 16, 64, 1, 3, (25, 17)), (13, 9, 128, 1, 1, (4, 4)), (12, 16, 512, 64, 37, (512, 512)),
            (8, 5, 256, 64, 3, (64, 64))]
    out += [(f, 16, 256, 16, 3, (512, 512)) for f in (12, 13, 14)]
    return out


GRID = _micro_grid()
GRID_IDS = [f"f{f}-d{d}-c{c}-hid{hid}-n{n}-hw{h}x{w}" for f, d, c, hid, n, (h, w) in GRID]


def micro_case(flags, d, c, hid, n, h, w):
    """Kernel inputs (fp32 on the device) and the plane-sum reference of one case."""
    from spff_b200._lib import Shape
    hw = h * w
    r = gen(flags * 7919 + d * 131 + c + hid * 17 + n * 3 + hw)
    S, R, coef, gamma = plane_inputs(r, n, c, d, hw)
    t = micro_params(r, c, d, hid)
    leaves = {k: v.clone().requires_grad_() for k, v in t.items()}
    se = se_dict(leaves["w1"], leaves["b1"], leaves["w2"], leaves["b2"])
    ref = plane_reference(S, R, hw, lambda x: tail64(x, flags, leaves["g1"], leaves["bt"], leaves["kfg"], se),
                          list(leaves.values()))
    ref["grads"] = dict(zip(leaves, ref["grads"]))
    dev = dict(S=cu(S), R=cu(R), coef=cu(coef), gamma=cu(gamma), shape=Shape(n, d, h, w),
               g1=cu(t["g1"]) if flags & EFILM else None, bt=cu(t["bt"]) if flags & EFILM else None,
               kfg=cu(t["kfg"]) if flags & FOURIER else None,
               se=tuple(cu(t[k]) for k in ("w1", "b1", "w2", "b2")) if flags & CHANSE else None)
    return dev, ref, dict(S=S, R=R, coef=coef, gamma=gamma, hw=hw, r=r)


@pytest.mark.parametrize("flags,d,c,hid,n,hw", GRID, ids=GRID_IDS)
def test_gate_micro_fwd(flags, d, c, hid, n, hw):
    """P and Q, each on its own, against the plane-sum reference."""
    from spff_b200 import ops
    dev, ref, _ = micro_case(flags, d, c, hid, n, *hw)
    P, Q = nan(n, d, c), nan(n, d, c)
    ops.gate_micro_fwd(dev["S"], dev["g1"], dev["bt"], dev["kfg"], dev["se"], flags, c, dev["shape"], P, Q)
    torch.cuda.synchronize()
    check("P", P, ref["P"])
    if flags & EFILM:
        check("Q", Q, ref["Q"])
    else:
        assert torch.equal(Q, torch.zeros_like(Q)), "Q of a block without EnergyFiLM is 0"


@pytest.mark.parametrize("flags,d,c,hid,n,hw", GRID, ids=GRID_IDS)
def test_gate_micro_bwd(flags, d, c, hid, n, hw):
    """Every output: bcoef (x = gamma rstd, y = mean dz, z = mean dz xhat, w = 0), dSa, Pout, and the accumulated
    dgamma, dbeta, dg1, dbt, dkfg, dse_w1, dse_b1, dse_w2, dse_b2. The same once for the whole batch and once as two
    sample groups accumulating into the same buffers. With flags 0 both routes: the InstanceNorm-only kernel (dSa and
    Pout NULL) and the gate kernel (dSa and Pout given). Accumulators of a gate the block does not have stay NaN."""
    from spff_b200 import ops
    from spff_b200._lib import Shape
    h, w = hw
    dev, ref, host = micro_case(flags, d, c, hid, n, h, w)
    hwf = float(h * w)
    rstd, gamma = host["coef"][..., 3], host["gamma"]
    want = {"bcoef": torch.stack([gamma * rstd, ref["sum_dz"] / (d * hwf), ref["sum_dzx"] / (d * hwf),
                                  torch.zeros_like(rstd)], dim=-1),
            "dSa": ref["dSa"], "Pout": ref["P"], "dgamma": ref["sum_dzx"].sum(0), "dbeta": ref["sum_dz"].sum(0)}
    acc_names = ["dgamma", "dbeta"]
    for k, leaf, bit in (("dg1", "g1", EFILM), ("dbt", "bt", EFILM), ("dkfg", "kfg", FOURIER), ("dse_w1", "w1", CHANSE),
                         ("dse_b1", "b1", CHANSE), ("dse_w2", "w2", CHANSE), ("dse_b2", "b2", CHANSE)):
        g = ref["grads"][leaf]
        shape = {"g1": (c, d), "bt": (c, d), "kfg": (d,), "w1": (hid, c), "b1": (hid,), "w2": (c, hid), "b2": (c,)}[leaf]
        if flags & bit:
            want[k] = g if g is not None else torch.zeros(shape, dtype=torch.float64)
            acc_names.append(k)
        else:
            want[k] = shape              # not owned: must stay NaN
    r = host["r"]
    init = {k: q32(r(*want[k].shape) * max(float(want[k].abs().max()), 1e-30)) for k in acc_names}

    routes = ["gates"] if flags else ["in_only", "gates"]
    splits = [[(0, n)]] + ([[(0, n // 2), (n // 2, n)]] if n > 1 else [])
    for route in routes:
        for split in splits:
            tag = f"[{route},{len(split)} group(s)]"
            out = {k: (cu(init[k]) if k in init else nan(*want[k])) for k in want if k not in ("bcoef", "dSa", "Pout")}
            bcoef = nan(n, c, 4)
            dSa = nan(n, d, c) if route == "gates" else None
            Pout = nan(n, d, c) if route == "gates" else None
            for s0, s1 in split:
                ops.gate_micro_bwd(dev["R"][s0:s1], dev["S"][s0:s1], dev["coef"][s0:s1], dev["gamma"], dev["g1"], dev["bt"],
                                   dev["kfg"], dev["se"], flags, c, Shape(s1 - s0, d, h, w), bcoef[s0:s1],
                                   dSa[s0:s1] if dSa is not None else None, Pout[s0:s1] if Pout is not None else None,
                                   out["dgamma"], out["dbeta"], out["dg1"], out["dbt"], out["dkfg"],
                                   (out["dse_w1"], out["dse_b1"], out["dse_w2"], out["dse_b2"]))
            torch.cuda.synchronize()
            bx, wx = bcoef[..., 0].double().cpu(), want["bcoef"][..., 0]
            assert float((bx - wx).abs().max()) <= U * float(wx.abs().max()), f"bcoef.x{tag}: gamma * rstd is one fp32 rounding"
            assert torch.equal(bcoef[..., 3], torch.zeros_like(bcoef[..., 3])), f"bcoef.w{tag} is 0"
            check(f"bcoef.y{tag}", bcoef[..., 1], want["bcoef"][..., 1])
            check(f"bcoef.z{tag}", bcoef[..., 2], want["bcoef"][..., 2])
            if route == "gates":
                if flags:
                    check(f"dSa{tag}", dSa, want["dSa"], floor=dsa_floor(host["R"], hwf))
                else:
                    assert torch.equal(dSa, torch.zeros_like(dSa)), f"dSa{tag}: a block without gates has no S gradient"
                check(f"Pout{tag}", Pout, want["Pout"])
            for k in out:
                if k in init:
                    check(f"{k}{tag}", out[k], want[k], tol=TOL_ACC, init=init[k])
                else:
                    untouched(f"{k}{tag}", out[k])


# --------------------------------------------------------------------------------------------------------------------
# 5. the configurations the variants run, through the engine's GateTables
# --------------------------------------------------------------------------------------------------------------------
STAGE = {"enc1": 0, "enc2": 1, "enc3": 2, "bott": 3}        # oracle.core_forward: SE stage of each encoder block


def oracle_block_tail(p, variant, b, x):
    """The gates of block b as oracle.core_forward composes them for `variant`, on fp64 parameters p."""
    from oracle import spff_oracle as O
    v = O.VARIANTS[variant]
    with fp64_oracle():
        if v["efilm"]:
            x = O._efilm(p, f"model.{b}.efilm", x)
        if v["fgate"]:
            x = O._fgate(p, f"model.{b}.fgate", x)
        if b in STAGE and v["se"]:
            x = O._channel_se(p, f"model.se.{STAGE[b]}", O._spectral_se(x))
    return x


def spct_variants():
    """(name, net_config, frames) of every SPCT variant in config.VARIANTS; frames = the 5 energy bins, padded to the
    variant's multiple (16 for SP_UNet)."""
    from innovative3D import config as C
    from innovative3D.models import UNet3D_SpectralCore
    out = []
    for name, builder, _, _ in C.VARIANTS[:len(C.B200_VARIANT_NAMES)]:
        lit = builder()
        if isinstance(lit.model, UNet3D_SpectralCore):
            m = getattr(lit, "_pad_multiple", 0)
            out.append((name, lit.model.net_config(), -(-C.NUM_FRAMES // m) * m if m else C.NUM_FRAMES))
    return out


def test_variant_configurations_through_gate_tables():
    """For every SPCT variant and block, with the variant's name-seeded weights: GateTables builds the tables,
    gate_micro_fwd / _bwd run as the engine calls them (flags from net_config().block_flags, channels, SE weight
    reshapes, the level's native plane size), and GateTables.finish() folds the table gradients into the EFiLM MLP and
    FourierGate parameters. Tables, P, Q, bcoef, dSa, Pout and every parameter gradient are compared with fp64 autograd
    through the oracle's block tail of that variant."""
    from oracle import spff_oracle as O
    from spff_b200 import engine
    from spff_b200._lib import Shape
    from spff_b200 import ops
    variants = spct_variants()
    assert {v[0] for v in variants} >= {"SPFF-UNet", "E_SP_UNet", "FG_SP_UNet", "SP_UNet", "PlainCore_UNet"}
    n = 3
    for vi, (variant, cfg, frames) in enumerate(variants):
        w64 = {k: v.double() for k, v in O.det_weights(O.param_shapes(variant, frames=frames)).items()}
        p32 = {k[len("model."):]: cu(v) for k, v in w64.items()}
        G = {k: torch.zeros_like(v) for k, v in p32.items()}
        T = engine.GateTables(cfg, p32, frames, need_grad=True)
        cn2 = cfg.conv_names[1]
        want = {}
        for b in engine.BLOCKS:
            c = cfg.channels(b)[1]
            flags = cfg.block_flags(b)
            where = f"{variant} {b} (flags {flags}, c {c}, F {frames})"
            side = 512 >> (engine._LEVEL[b] - 1)
            hw = side * side
            r = gen(50 + 10 * vi + engine.BLOCKS.index(b))
            S, R, coef, _ = plane_inputs(r, n, c, frames, hw)
            gname, bname = f"{b}.{cn2}.1.weight", f"{b}.{cn2}.1.bias"
            leaves = {k: v.clone().requires_grad_() for k, v in w64.items()
                      if k.startswith((f"model.{b}.efilm.", f"model.{b}.fgate.")) or
                      (b in STAGE and k.startswith(f"model.se.{STAGE[b]}."))}
            p = {**w64, **leaves}
            ref = plane_reference(S, R, hw, lambda x: oracle_block_tail(p, variant, b, x), list(leaves.values()))
            for k, g in zip(leaves, ref["grads"]):
                want[k[len("model."):]] = g if g is not None else torch.zeros_like(leaves[k])
            gamma = w64[f"model.{gname}"]
            want[gname], want[bname] = ref["sum_dzx"].sum(0), ref["sum_dz"].sum(0)
            if cfg.efilm or cfg.fgate:
                g1, bt, kfg = ref_tables({k.replace(f"model.{b}.efilm.", "e.").replace(f"model.{b}.fgate.", "f."): v
                                          for k, v in w64.items()}, c, frames, cfg.efilm, cfg.fgate)
                for name, got, ref_t in (("g1", T.g1[b], g1), ("bt", T.bt[b], bt), ("kfg", T.kfg[b], kfg)):
                    if ref_t is not None:
                        check(f"table {name}[{where}]", got, ref_t)
            shp = Shape(n, frames, side, side)
            Sd, Rd, coefd = cu(S), cu(R), cu(coef)
            if flags:
                P, Q = nan(n, frames, c), nan(n, frames, c)
                ops.gate_micro_fwd(Sd, T.g1[b], T.bt[b], T.kfg[b], T.se[b], flags, c, shp, P, Q)
                check(f"P[{where}]", P, ref["P"])
                if cfg.efilm:
                    check(f"Q[{where}]", Q, ref["Q"])
                else:
                    assert torch.equal(Q, torch.zeros_like(Q)), f"Q[{where}] of a block without EnergyFiLM is 0"
            dse = None
            if flags & CHANSE:
                i = STAGE[b]
                dse = (G[f"se.{i}.fc.0.weight"].view(-1, c), G[f"se.{i}.fc.0.bias"], G[f"se.{i}.fc.2.weight"].view(c, -1),
                       G[f"se.{i}.fc.2.bias"])
            bcoef = nan(n, c, 4)
            dSa = nan(n, frames, c) if flags else None
            Pout = nan(n, frames, c) if flags else None
            ops.gate_micro_bwd(Rd, Sd if flags else None, coefd, p32[gname], T.g1[b], T.bt[b], T.kfg[b], T.se[b], flags, c,
                               shp, bcoef, dSa, Pout, G[gname], G[bname], T.dg1[b], T.dbt[b], T.dkfg[b], dse)
            cnt = frames * float(hw)
            check(f"bcoef.y[{where}]", bcoef[..., 1], ref["sum_dz"] / cnt)
            check(f"bcoef.z[{where}]", bcoef[..., 2], ref["sum_dzx"] / cnt)
            check(f"bcoef.x[{where}]", bcoef[..., 0], gamma * coef[..., 3], tol=U)
            if flags:
                check(f"dSa[{where}]", dSa, ref["dSa"], floor=dsa_floor(R, hw))
                check(f"Pout[{where}]", Pout, ref["P"])
        T.finish(G)
        torch.cuda.synchronize()
        for k, g in want.items():
            check(f"grad {k}[{variant}]", G[k], g, tol=TOL_ACC)
        for k, g in G.items():
            if k not in want:
                assert not g.any(), f"{variant}: {k} is not a gate or norm parameter of the blocks but got a gradient"


# --------------------------------------------------------------------------------------------------------------------
# 6. refusals
# --------------------------------------------------------------------------------------------------------------------
REFUSE_MICRO = [
    ("d=0", dict(flags=15, d=0, hid=4)), ("d=17", dict(flags=15, d=17, hid=4)),
    ("hid=0", dict(flags=CHANSE, d=5, hid=0)), ("hid=65", dict(flags=CHANSE | SPECSE, d=16, hid=65)),
    ("efilm-without-g1", dict(flags=EFILM, d=5, hid=4, drop=("g1",))),
    ("efilm-without-bt", dict(flags=EFILM | FOURIER, d=8, hid=4, drop=("bt",))),
    ("fourier-without-kfg", dict(flags=FOURIER, d=5, hid=4, drop=("kfg",))),
    ("chanse-without-fc", dict(flags=CHANSE | SPECSE, d=5, hid=4, drop=("w1", "b1", "w2", "b2"))),
]


@pytest.mark.parametrize("which", ["fwd", "bwd"])
@pytest.mark.parametrize("case", REFUSE_MICRO, ids=[k for k, _ in REFUSE_MICRO])
def test_gate_micro_refuses(case, which):
    """A bin count outside 1..16, an SE width outside 1..64 with ChannelSE, or a gate flag without its tables or fc
    weights raises RuntimeError, and nothing is written. The C entry points are called directly, so that the SE width
    is passed as given whatever the weights' shape."""
    from spff_b200._lib import Shape, call, ptr, stream_ptr
    kw = case[1]
    flags, d, hid, c, n = kw["flags"], kw["d"], kw["hid"], 64, 2
    dd = max(d, 1)                # buffers with room for the bins the call names
    r = gen(9)
    S, R, coef, gamma = (cu(t) for t in plane_inputs(r, n, c, dd, 16))
    t = {k: (None if k in kw.get("drop", ()) else cu(v)) for k, v in micro_params(r, c, dd, 4).items()}
    shp = Shape(n, d, 4, 4)
    weights = [ptr(t[k]) for k in ("g1", "bt", "kfg", "w1", "b1", "w2", "b2")]
    if which == "fwd":
        outs = [nan(n, dd, c), nan(n, dd, c)]
        with pytest.raises(RuntimeError, match="gate_micro"):
            call("spff_gate_micro_fwd", ptr(S), *weights, hid, flags, c, shp, *(ptr(o) for o in outs), stream_ptr())
    else:
        outs = [nan(n, c, 4), nan(n, dd, c), nan(n, dd, c), nan(c), nan(c), nan(c, dd), nan(c, dd), nan(dd),
                nan(4, c), nan(4), nan(c, 4), nan(c)]
        with pytest.raises(RuntimeError, match="gate_micro"):
            call("spff_gate_micro_bwd", ptr(R), ptr(S), ptr(coef), ptr(gamma), *weights, hid, flags, c, shp,
                 *(ptr(o) for o in outs), stream_ptr())
    torch.cuda.synchronize()
    for i, o in enumerate(outs):
        untouched(f"output {i}", o)


@pytest.mark.parametrize("which", ["fwd", "bwd"])
@pytest.mark.parametrize("frames", [0, 17])
def test_gate_tables_refuse(frames, which):
    """frames outside 1..16 raises RuntimeError, and nothing is written."""
    from spff_b200 import ops
    c = 32
    p = table_params(gen(11), c, 16)
    p["f.freq_mask"] = q32(1 + 0.2 * gen(12)(1, 1, frames // 2 + 1, 1, 1))
    args = table_args(p, True, True)
    f = max(frames, 1)
    if which == "fwd":
        outs = [nan(c, f), nan(c, f), nan(f)]
        with pytest.raises(RuntimeError, match="gate_tables_fwd"):
            ops.gate_tables_fwd(*args, c, frames, *outs)
    else:
        outs = [nan(32, 16, 1), nan(32), nan(2 * c, 32, 1), nan(2 * c), nan(frames // 2 + 1), nan(1)]
        with pytest.raises(RuntimeError, match="gate_tables_bwd"):
            ops.gate_tables_bwd(*args, c, frames, cu(torch.ones(c, f)), cu(torch.ones(c, f)), cu(torch.ones(f)), *outs)
    torch.cuda.synchronize()
    for i, o in enumerate(outs):
        untouched(f"output {i}", o)
