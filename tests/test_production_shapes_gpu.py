"""GPU: the step's kernels at the layouts and sizes the engine runs them.

1. A recorder wraps every public function of `spff_b200.ops` while SPFF-UNet and PlainCore_UNet run `fit_step`,
   `predict_labels` and `eval_step` on one native 512 x 512 slice and on one 200 x 136 slice (whose level-3 and
   level-4 planes do not tile by 16 x 8). Each call leaves a signature: the entry point, the shape, dtype, strides and
   channel offset of every tensor argument, and the scalar arguments. `ENTRY_POINTS` gives every entry point either a
   reference or the reason it is not replayed; an entry point the step calls without being listed there fails.
2. Every distinct signature is replayed on fresh random inputs of the same shape, pitch and channel offset (a concat
   half is a slice of a NaN-filled wider buffer), with every output NaN-filled first, and compared with a plain
   high-precision reference. Besides the rel-L2 bounds of the other kernel tests:
   - per tile: for every block of 128 positions x 32 channels, max |kernel - reference| <= one bf16 ulp of the block's
     largest reference value (the output's own rounding) + the accumulation term stated with each entry point;
   - no stray writes: no NaN is left in an output, and the channels of a shared buffer the call does not own keep
     their NaN bit pattern;
   - the statistics slots the halo-tile conv kernel does not fill read exactly 0.
   Reductions (statistics, weight gradients) are compared element by element with a probabilistic bound on fp32
   summation (Higham & Mary, SIAM J. Sci. Comput. 41(5), 2019): summing N terms in any order in fp32 errs by at most
   lambda * sqrt(N) * u * sum|terms| with probability >= 1 - 2 exp(-lambda^2 / 2); lambda = 6 (u = 2^-24).
3. Level-1 entry points on a group of 52 slices of 5 x 512 x 512, where the concat buffers (pitch 64) hold 4.4e9
   elements, past 2^32: samples 0, n/2 and n-1 are checked against references computed on them alone, and batch
   reductions against the fp64 sum of per-sample references. Every sample gets its own random content.
"""
import inspect
import math
import time

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

U = 2.0 ** -24                  # fp32 unit roundoff
LAMBDA = 6.0                    # probabilistic summation bound: failure probability 2 exp(-18) ~ 3e-8 per element
K = 13
IGN = 255
WORST = {}                      # entry point -> worst per-tile error / bound seen


def gamma(k):
    """Worst-case relative error of a k-term fp32 dot product (Higham, Accuracy and Stability, eq. 3.4)."""
    return k * U / (1 - k * U)


def sum_bound(abs_sum, n):
    return LAMBDA * math.sqrt(n) * U * abs_sum


def sum_rel_bound(n):
    """rel-L2 bound of a gradient summed over n positions in fp32 (the weight gradients). The tensor cores accumulate in
    fp32 without round-to-nearest (they truncate: Fasi, Higham, Mikaitis & Pranesh, PeerJ Comput. Sci. 7:e330, 2021),
    so each addition errs by delta * S with |delta| < 2u, where S is the partial sum it produces; model the deltas as
    independent. In any summation order each partial sum adds at most n independent zero-mean terms, so
    E[S^2] <= n sigma^2, and over n - 1 additions E[err^2] <= 4 u^2 n^2 sigma^2 against E[dw^2] = n sigma^2: an rms
    relative error <= 2 u sqrt(n). The rel-L2 pools thousands of weights, so it estimates that rms closely; asserted
    with a factor 2, and never below the 1e-4 of test_conv3_gpu.py. At a 52-slice group (n = 6.8e7) that is 2e-3, while
    one sample read from the wrong place shows as 0.2."""
    return max(1e-4, 4 * U * math.sqrt(n))


def _nan16():
    return int(torch.tensor(float("nan"), dtype=torch.bfloat16).view(torch.int16))


# --------------------------------------------------------------------------------------------------------------------
# buffers and checks
# --------------------------------------------------------------------------------------------------------------------
class PM:
    """A bf16 position-major view [n, d, h, w, c] at channel offset `off` of a NaN-filled buffer of pitch `ld`."""

    def __init__(self, n, d, h, w, c, ld=None, off=0):
        self.ld = ld or c
        self.c, self.off = c, off
        self.base = torch.full((n, d, h, w, self.ld), float("nan"), dtype=torch.bfloat16, device="cuda")
        self.t = self.base[..., off:off + c]

    @classmethod
    def of(cls, ts):
        _, shape, _, strides, off = ts
        return cls(*shape, ld=strides[3], off=off)

    def fill(self, g, scale=1.0, shift=0.0):
        """Random content, drawn sample by sample so that every sample differs."""
        for i in range(self.t.shape[0]):
            self.t[i] = (torch.randn(self.t.shape[1:], generator=g, device="cuda") * scale + shift).to(torch.bfloat16)
        return self

    def ncdhw(self, i, dtype=torch.float32):
        return self.t[i:i + 1].permute(0, 4, 1, 2, 3).to(dtype)

    def check_written(self, what):
        """Every owned element written (no NaN left), every other channel of the buffer untouched."""
        nan16 = _nan16()
        for i in range(self.t.shape[0]):
            assert not bool(torch.isnan(self.t[i]).any()), f"{what}: sample {i} has elements the kernel did not write"
            for rest in (self.base[i, ..., :self.off], self.base[i, ..., self.off + self.c:]):
                if rest.shape[-1]:
                    assert bool((rest.view(torch.int16) == nan16).all()), \
                        f"{what}: sample {i}: the call wrote channels of the shared buffer it does not own"


def tile_check(entry, got, ref, extra, sample=0):
    """got / ref [1, C, d, h, w] fp32, extra (tensor of that shape or a float): the accumulation term per element.
    For every tile of 128 positions (flattened d, h, w) x 32 channels: max|got - ref| <= ulp_bf16(max|ref|) + max(extra)."""
    c = ref.shape[1]
    flat = lambda t: t.permute(0, 2, 3, 4, 1).reshape(-1, c)
    err, mag = flat((got - ref).abs()), flat(ref.abs())
    ext = flat(extra) if torch.is_tensor(extra) else torch.full_like(mag, float(extra))
    p = mag.shape[0]
    pad = (-p) % 128
    if pad:
        err, mag, ext = (F.pad(t, (0, 0, 0, pad)) for t in (err, mag, ext))
    shp = (mag.shape[0] // 128, 128, c // 32, 32)
    err, mag, ext = (t.reshape(shp).amax(dim=(1, 3)) for t in (err, mag, ext))
    _, ex = torch.frexp(mag)
    ulp = torch.where(mag > 0, torch.ldexp(torch.ones_like(mag), ex - 8), torch.zeros_like(mag))
    bound = ulp + ext
    ratio = _ratio(err, bound)
    worst = int(ratio.argmax())
    t, cb = divmod(worst, c // 32)
    r = float(ratio.reshape(-1)[worst])
    WORST[entry] = max(WORST.get(entry, 0.0), r)
    d, h, w = ref.shape[2:]
    pos = t * 128
    where = f"sample {sample}, tile {t} (d={pos // (h * w)}, h={pos // w % h}, w={pos % w}), channels {32 * cb}..{32 * cb + 31}"
    assert bool((err <= bound).all()), \
        f"{entry}: {where}: max error {float(err.reshape(-1)[worst]):.3e} > bound {float(bound.reshape(-1)[worst]):.3e}"
    return r


def _ratio(err, bound):
    inf = torch.full_like(err, float("inf"))
    return torch.where(bound > 0, err / bound.clamp(min=1e-300), torch.where(err > 0, inf, torch.zeros_like(err)))


def rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-300))


def elem_check(entry, got, ref, bound):
    """Element-wise |got - ref| <= bound (reductions); records the worst ratio."""
    err = (got.double() - ref.double()).abs()
    bound = bound.double() if torch.is_tensor(bound) else torch.full_like(err, float(bound))
    ratio = _ratio(err, bound)
    i = int(ratio.argmax())
    r = float(ratio.reshape(-1)[i])
    WORST[entry] = max(WORST.get(entry, 0.0), r)
    assert bool((err <= bound).all()), f"{entry}: element {i}: error {float(err.reshape(-1)[i]):.3e} > bound " \
                                       f"{float(bound.reshape(-1)[i]):.3e}"


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


def _dtype(ts):
    return getattr(torch, ts[2])


def _nanlike(ts):
    return torch.full(ts[1], float("nan"), dtype=_dtype(ts), device="cuda")


def _labels(ts, g, ignore):
    """Classes 0..K-1 with 5 % ignore_index, drawn sample by sample."""
    lab = torch.empty(ts[1], dtype=_dtype(ts), device="cuda")
    for i in range(lab.shape[0]):
        li = torch.randint(0, K, lab.shape[1:], generator=g, device="cuda", dtype=lab.dtype)
        li[torch.rand(lab.shape[1:], generator=g, device="cuda") < 0.05] = ignore
        lab[i] = li
    return lab


def _halo_runs(kernel, h, w, gemm_k):
    """conv3_halo_applicable (conv3_halo.cu) for depth 5: planes tiling by 16 x 8, and K = 32 or >= 128 unless forced."""
    if kernel == "rows" or h % 16 or w % 8:
        return False
    return kernel == "halo" or gemm_k == 32 or gemm_k >= 128


# --------------------------------------------------------------------------------------------------------------------
# replays: a = {argument name: signature}; per-position outputs are checked on `samples`, reductions on every sample
# --------------------------------------------------------------------------------------------------------------------
def _check_partials(entry, partial, refs, abs_err, n_slot, halo, shape, c):
    """partial [n, slots, 2, c] of one conv output: slot sums == fp64 sums of the reference output within the per-element
    error of the output (abs_err) plus fp32 summation of n_slot terms per slot; unfilled halo slots exactly 0."""
    i, ref = refs
    tot = partial[i].double().sum(0)                                     # [2, c]
    r = ref.double()
    want = torch.stack([r.sum(dim=(0, 2, 3, 4)), (r * r).sum(dim=(0, 2, 3, 4))])
    e = abs_err.double()
    b1 = e.sum(dim=(0, 2, 3, 4)) + sum_bound(r.abs().sum(dim=(0, 2, 3, 4)), n_slot)
    b2 = ((2 * r.abs() + e) * e).sum(dim=(0, 2, 3, 4)) + sum_bound((r * r).sum(dim=(0, 2, 3, 4)), n_slot)
    elem_check(entry + " partials", tot, want, torch.stack([b1, b2]) * 1.0001 + 1e-30)
    if halo:
        _, d, h, w = shape
        mine = (h // 16) * (w // 8) * ((d + 4) // 5)
        rest = partial[i, mine:]
        assert bool((rest == 0).all()), f"{entry}: statistics slots {mine}.. of sample {i} are not zero"


def replay_conv(entry, a, samples, kernel):
    """conv3d_k3_fwd(_stats) / dgrad(_stats) against F.conv3d / F.conv_transpose3d in fp64 on the bf16-rounded operands
    (the fp32 reference with TF32 off, without its own rounding). Accumulation term: the kernel sums K = 27 * C_in(GEMM)
    exact bf16 products in fp32, within gamma(K) * sum|products| of the exact value: gamma(K) * (|x| conv |w|)."""
    from spff_b200 import ops
    from spff_b200._lib import Shape
    fwd = entry.startswith("conv3d_k3_fwd")
    xa, ya = (a["x"], a["y"]) if fwd else (a["dy"], a["dx"])
    cin, cout = (a["cin"], a["cout"]) if fwd else (a["cout"], a["cin"])    # GEMM input / output channels
    g = _gen(11)
    x = PM.of(xa).fill(g)
    y = PM.of(ya)
    n, d, h, w, _ = y.t.shape
    wt = torch.randn(cout, cin, 3, 3, 3, generator=g, device="cuda") / math.sqrt(27 * cin)   # as (out, in) of the GEMM
    if fwd:
        wf, _ = ops.pack_conv3_weight(wt)
    else:                                           # dgrad of the conv whose weight is [cin_conv = cout, cout_conv = cin]
        _, wf = ops.pack_conv3_weight(wt.transpose(0, 1).contiguous())
    stats = a.get("partial") is not None
    partial = _nanlike(a["partial"]) if stats else None
    args = (x.t, cin, wf, y.t, cout) + ((partial,) if stats else ())
    getattr(ops, entry)(*args)
    torch.cuda.synchronize()
    y.check_written(entry)
    if stats:
        assert not bool(torch.isnan(partial).any()), f"{entry}: statistics slots left unwritten"
    wq = wt.to(torch.bfloat16).double()
    worst = 0.0
    for i in samples:
        xi = x.ncdhw(i, torch.float64)
        if fwd:
            ref = F.conv3d(xi, wq, padding=1)
            absr = F.conv3d(xi.abs(), wq.abs(), padding=1)
        else:
            wt_t = wq.transpose(0, 1)               # conv weight [cout_conv, cin_conv] -> its transposed conv
            ref = F.conv_transpose3d(xi, wt_t, padding=1)
            absr = F.conv_transpose3d(xi.abs(), wt_t.abs(), padding=1)
        got = y.ncdhw(i)
        extra = (gamma(27 * cin) * absr).float()
        ref64, ref = ref, ref.float()
        worst = max(worst, tile_check(entry, got, ref, extra, i))
        assert rel(got, ref) < 4e-3
        if stats:
            slots = partial.shape[1]
            n_slot = -(-d * h * w // slots) + 8
            _check_partials(entry, partial, (i, ref64), extra, n_slot, _halo_runs(kernel, h, w, cin),
                            (n, d, h, w), cout)
        del xi, ref, ref64, absr, got, extra
    return worst


def replay_conv3d_k3_wgrad(a, samples):
    """dw = beta * dw0 + sum over positions of x (x) dy: the fp64 sum of per-sample conv3d_weight references. Bound per
    weight: fp32 summation of N = n*d*h*w exact bf16 products, plus the rounding of beta*dw0; and the rel-L2 1e-4 of
    test_conv3_gpu.py."""
    from spff_b200 import ops
    cin, cout, beta = a["cin"], a["cout"], a["beta"]
    g = _gen(12)
    x = PM.of(a["x"]).fill(g)
    dy = PM.of(a["dy"]).fill(g)
    dw0 = torch.randn(cout, cin, 3, 3, 3, generator=g, device="cuda")
    dw = dw0.clone()
    ops.conv3d_k3_wgrad(x.t, cin, dy.t, cout, dw, beta)
    torch.cuda.synchronize()
    assert bool(torch.isfinite(dw).all())
    ref = beta * dw0.double()
    absr = torch.zeros_like(ref)
    for i in range(x.t.shape[0]):
        xi, dyi = x.ncdhw(i, torch.float64), dy.ncdhw(i, torch.float64)
        ref += torch.nn.grad.conv3d_weight(xi, dw.shape, dyi, padding=1)
        absr += torch.nn.grad.conv3d_weight(xi.abs(), dw.shape, dyi.abs(), padding=1)
    n, d, h, w, _ = x.t.shape
    elem_check("conv3d_k3_wgrad", dw, ref, sum_bound(absr, n * d * h * w) + 2 * U * (beta * dw0.abs().double()) + 1e-30)
    r = rel(dw - beta * dw0, ref - beta * dw0.double())
    print(f"conv3d_k3_wgrad {n}x{d}x{h}x{w} {cin}->{cout}: rel-L2 {r:.2e}")
    assert r < sum_rel_bound(n * d * h * w), r


def replay_conv3d_stem_fwd_stats(a, samples):
    """Stem forward (Cin = 1) against F.conv3d in fp64 on the fp32 input. The kernel multiplies bf16 hi + lo splits of
    x and w (three products, fp32 accumulation): each operand keeps a 2^-16 relative error and lo*lo is dropped, so
    <= 3 * 2^-16 * sum|x w| + 2 gamma(27) * sum|x w| <= 2^-14 * (|x| conv |w|)."""
    from spff_b200 import ops
    g = _gen(13)
    xs = a["x"][1]
    x = torch.randn(xs, generator=g, device="cuda")
    wt = torch.randn(a["w"][1], generator=g, device="cuda") * 0.2
    y = PM.of(a["y"])
    partial = _nanlike(a["partial"])
    ops.conv3d_stem_fwd_stats(x, wt, y.t, a["cout"], partial)
    torch.cuda.synchronize()
    y.check_written("conv3d_stem_fwd_stats")
    assert not bool(torch.isnan(partial).any())
    n, d, h, w, _ = y.t.shape
    w64 = wt.double()
    for i in samples:
        xi = x[i:i + 1].double()
        ref = F.conv3d(xi, w64, padding=1)
        extra = (2.0 ** -14 * F.conv3d(xi.abs(), w64.abs(), padding=1)).float()
        tile_check("conv3d_stem_fwd_stats", y.ncdhw(i), ref.float(), extra, i)
        n_slot = -(-d * h * w // partial.shape[1]) + 8
        _check_partials("conv3d_stem_fwd_stats", partial, (i, ref), extra, n_slot, False, (n, d, h, w), a["cout"])


def replay_conv3d_stem_wgrad(a, samples):
    """Stem weight gradient: exact bf16(x) * bf16(dy) products summed in fp32 (test_kernels_gpu.py::test_stem)."""
    from spff_b200 import ops
    g = _gen(14)
    x = torch.randn(a["x"][1], generator=g, device="cuda")
    dy = PM.of(a["dy"]).fill(g)
    beta = a["beta"]
    dw0 = torch.randn(a["dw"][1], generator=g, device="cuda")
    dw = dw0.clone()
    ops.conv3d_stem_wgrad(x, dy.t, a["cout"], dw, beta)
    torch.cuda.synchronize()
    ref = beta * dw0.double()
    absr = torch.zeros_like(ref)
    for i in range(x.shape[0]):
        xi = x[i:i + 1].to(torch.bfloat16).double()
        dyi = dy.ncdhw(i, torch.float64)
        ref += torch.nn.grad.conv3d_weight(xi, dw.shape, dyi, padding=1)
        absr += torch.nn.grad.conv3d_weight(xi.abs(), dw.shape, dyi.abs(), padding=1)
    elem_check("conv3d_stem_wgrad", dw, ref, sum_bound(absr, x.numel()) + 2 * U * beta * dw0.abs().double() + 1e-30)
    r = rel(dw - beta * dw0, ref - beta * dw0.double())
    print(f"conv3d_stem_wgrad {tuple(x.shape)}: rel-L2 {r:.2e}")
    assert r < sum_rel_bound(x.numel()), r


def replay_in_coeffs_from_partials(a, samples):
    """coef = {A, B, mean, rstd} from fp32 partials: fp64 reference; the kernel sums in double and rounds the results
    to fp32, so a few fp32 roundings (2^-20 relative, of |beta| + |mean A| for B)."""
    from spff_b200 import ops
    g = _gen(15)
    n, slots, _, c = a["partial"][1]
    count, eps = a["count"], a["eps"]
    m = count / slots
    s1 = torch.randn(n, slots, c, generator=g, device="cuda") * math.sqrt(m) + 0.3 * m
    s2 = m * (1.2 + torch.rand(n, slots, c, generator=g, device="cuda")) + s1 * s1 / m
    partial = torch.stack([s1, s2], dim=2).contiguous()
    gm = torch.rand(c, generator=g, device="cuda") + 0.5
    bt = torch.randn(c, generator=g, device="cuda")
    coef = _nanlike(a["coef"])
    ops.in_coeffs_from_partials(partial, a["slots"], gm, bt, eps, n, c, count, coef)
    torch.cuda.synchronize()
    p = partial.double()
    mean = p[:, :, 0].sum(1) / count
    var = p[:, :, 1].sum(1) / count - mean * mean
    rstd = 1.0 / torch.sqrt(var + eps)
    A = rstd * gm.double()
    B = bt.double() - mean * A
    tol = 2.0 ** -20
    elem_check("in_coeffs_from_partials", coef[..., 0], A, tol * A.abs())
    elem_check("in_coeffs_from_partials", coef[..., 1], B, tol * (bt.double().abs() + (mean * A).abs()))
    elem_check("in_coeffs_from_partials", coef[..., 2], mean, tol * (mean.abs() + var.sqrt()))
    elem_check("in_coeffs_from_partials", coef[..., 3], rstd, tol * rstd)


def _coef_for(n, c, g):
    """{A, B, mean, rstd} of an InstanceNorm with gamma in [0.5, 1.5), beta ~ N(0, 0.3) on unit-scale inputs."""
    mean = torch.randn(n, c, generator=g, device="cuda") * 0.2
    rstd = 0.8 + 0.4 * torch.rand(n, c, generator=g, device="cuda")
    gm = 0.5 + torch.rand(n, c, generator=g, device="cuda")
    bt = 0.3 * torch.randn(n, c, generator=g, device="cuda")
    A = rstd * gm
    return torch.stack([A, bt - mean * A, mean, rstd], dim=-1).contiguous(), gm, bt


def _bc(t, i):     # per-(sample, channel) [n, c] -> [1, c, 1, 1, 1]
    return t[i].view(1, -1, 1, 1, 1)


def _bdc(t, i):    # per-(sample, plane, channel) [n, d, c] -> [1, c, d, 1, 1]
    return t[i].transpose(0, 1).reshape(1, -1, t.shape[1], 1, 1)


def _act(x, coef, i, slope):
    """z = x*A + B (fp32, as the kernels), m = lrelu'(z), a = lrelu(z), and the bound of z's own rounding."""
    A, B = _bc(coef[..., 0], i), _bc(coef[..., 1], i)
    z = x * A + B
    m = torch.where(z > 0, torch.ones_like(z), torch.full_like(z, slope))
    return z, m, z * m, 2 * U * ((x * A).abs() + B.abs())


def replay_norm_act_apply(a, samples):
    """y = lrelu(x*A + B): fp32 formula; accumulation term: z's two roundings on either side."""
    from spff_b200 import ops
    g = _gen(16)
    x = PM.of(a["x"]).fill(g)
    y = PM.of(a["y"])
    c, slope = a["c"], a["slope"]
    coef, _, _ = _coef_for(x.t.shape[0], c, g)
    ops.norm_act_apply(x.t, coef, y.t, c, slope)
    torch.cuda.synchronize()
    y.check_written("norm_act_apply")
    for i in samples:
        _, _, ref, ez = _act(x.ncdhw(i), coef, i, slope)
        tile_check("norm_act_apply", y.ncdhw(i), ref, 2 * ez, i)


def replay_norm_act_reduce(a, samples):
    """S[n, d, c] = sum over (h, w) of lrelu(x*A + B): fp64 sum of the fp32 terms; fp32 summation of h*w terms plus
    the terms' own rounding."""
    from spff_b200 import ops
    g = _gen(17)
    x = PM.of(a["x"]).fill(g)
    c, slope = a["c"], a["slope"]
    coef, _, _ = _coef_for(x.t.shape[0], c, g)
    S = _nanlike(a["S"]) if a["fixed_order"] else torch.zeros(a["S"][1], device="cuda")
    ops.norm_act_reduce(x.t, coef, S, c, slope, fixed_order=a["fixed_order"])
    torch.cuda.synchronize()
    _, _, h, w, _ = x.t.shape
    for i in range(x.t.shape[0]):
        _, _, act, ez = _act(x.ncdhw(i), coef, i, slope)
        ref = act.double().sum(dim=(3, 4))[0].t()                       # [d, c]
        b = sum_bound(act.abs().double().sum(dim=(3, 4))[0].t(), h * w) + 2 * ez.double().sum(dim=(3, 4))[0].t()
        elem_check("norm_act_reduce", S[i], ref, b)


def replay_norm_act_affine_apply(a, samples):
    """y = lrelu(x*A + B) * P + Q (fp32 formula; accumulation term: the roundings of z, a*P and + Q on either side),
    its (1,2,2) max-pool == the pool of the kernel's own y, the arg-max codes == the first maximum of its windows."""
    from spff_b200 import ops
    g = _gen(18)
    x = PM.of(a["x"]).fill(g)
    y = PM.of(a["y"])
    c, slope = a["c"], a["slope"]
    n, d, h, w, _ = x.t.shape
    coef, _, _ = _coef_for(n, c, g)
    P = Q = None
    if a["P"] is not None:
        P = 1 + 0.3 * torch.randn(n, d, c, generator=g, device="cuda")
        Q = 0.2 * torch.randn(n, d, c, generator=g, device="cuda")
    yp = PM.of(a["ypool"]) if a["ypool"] is not None else None
    codes = torch.full(a["pool_argmax"][1], 255, dtype=torch.uint8, device="cuda") if a["pool_argmax"] is not None else None
    ops.norm_act_affine_apply(x.t, coef, P, Q, y.t, yp.t if yp else None, c, slope, pool_argmax=codes)
    torch.cuda.synchronize()
    y.check_written("norm_act_affine_apply")
    if yp is not None:
        yp.check_written("norm_act_affine_apply pool")
    for i in samples:
        _, _, act, ez = _act(x.ncdhw(i), coef, i, slope)
        ref, extra = act, 2 * ez
        if P is not None:
            ref = act * _bdc(P, i) + _bdc(Q, i)
            extra = (2 * ez + 2 * U * act.abs()) * _bdc(P, i).abs() + 2 * U * ref.abs()
        tile_check("norm_act_affine_apply", y.ncdhw(i), ref, extra, i)
        if yp is not None:
            yi = y.t[i]                                                   # [d, h, w, c] bf16
            win = yi.reshape(d, h // 2, 2, w // 2, 2, c).permute(0, 1, 3, 5, 2, 4).reshape(d, h // 2, w // 2, c, 4)
            assert torch.equal(yp.t[i], win.amax(-1)), f"norm_act_affine_apply: pool of sample {i}"
            if codes is not None:
                first = win.float().argmax(-1).to(torch.uint8)            # first maximum, corner 2*kh + kw
                assert torch.equal(codes[i], first), f"norm_act_affine_apply: arg-max codes of sample {i}"


def replay_norm_act_bwd_reduce(a, samples):
    """R[n, d, c, 6] = per-plane sums of {dout*a, dout, dout*m, m, dout*m*xhat, m*xhat} (plain: slots 2 and 4 only, the
    others untouched). fp64 sums of the fp32 terms. The lean first stage derives slots 4 and 5 from the others
    ((sum dout*a - beta*sum dout*m)/gamma, (S - beta*sum m)/gamma), so their bound carries those sums' errors / gamma."""
    from spff_b200 import ops
    g = _gen(19)
    dout = PM.of(a["dout"]).fill(g)
    x = PM.of(a["x"]).fill(g)
    c, slope, plain, fixed = a["c"], a["slope"], a["plain"], a["fixed_order"]
    n, d, h, w, _ = x.t.shape
    coef, gm, bt = _coef_for(n, c, g)
    red = lambda t: t.double().sum(dim=(3, 4))[0].t()                    # [1, c, d, h, w] -> [d, c]

    def terms(i):
        xi = x.ncdhw(i)
        _, m, act, ez = _act(xi, coef, i, slope)
        xhat = (xi - _bc(coef[..., 2], i)) * _bc(coef[..., 3], i)
        return dout.ncdhw(i), m, act, xhat, ez
    S = None
    if a["S"] is not None:
        S = torch.stack([red(terms(i)[2]) for i in range(n)]).float().contiguous()
    R = _nanlike(a["R"]) if fixed else torch.zeros(a["R"][1], device="cuda")
    ops.norm_act_bwd_reduce(dout.t, x.t, coef, R, c, slope, plain=plain, fixed_order=fixed, S=S)
    torch.cuda.synchronize()
    produced = (2, 4) if plain else range(6)
    for i in range(n):
        do, m, act, xhat, ez = terms(i)
        sums = [do * act, do, do * m, m, do * m * xhat, m * xhat]
        gi, bi = gm[i].double().view(1, -1), bt[i].double().view(1, -1).abs()
        for j in range(6):
            got = R[i, ..., j]
            if j not in produced:
                untouched = torch.isnan(got) if fixed else got == 0
                assert bool(untouched.all()), f"norm_act_bwd_reduce: slot {j} written in plain mode"
                continue
            b = sum_bound(red(sums[j].abs()), h * w) + red(2 * ez * do.abs() if j in (0, 4) else 2 * ez)
            if j == 4:
                b = b + (sum_bound(red((do * act).abs()) + bi * red((do * m).abs()), h * w)
                         + red(2 * ez * do.abs())) / gi
            if j == 5:
                b = b + (sum_bound(red(act.abs()) + bi * red(m), h * w) + red(2 * ez)) / gi
            elem_check("norm_act_bwd_reduce", got, red(sums[j]), b * 1.0001 + 1e-30)
        del do, m, act, xhat, ez, sums


def replay_norm_act_bwd_apply(a, samples):
    """dx = c1 * (dz - c2 - xhat * c3), dz = (dout * P + dSa) * m: fp32 formula; accumulation term: the roundings of
    each term on either side (4 u of each magnitude, times |c1|)."""
    from spff_b200 import ops
    g = _gen(20)
    dout = PM.of(a["dout"]).fill(g)
    x = PM.of(a["x"]).fill(g)
    dx = PM.of(a["dx"])
    c, slope = a["c"], a["slope"]
    n, d, h, w, _ = x.t.shape
    coef, _, _ = _coef_for(n, c, g)
    bcoef = torch.stack([coef[..., 0], 0.1 * torch.randn(n, c, generator=g, device="cuda"),
                         0.1 * torch.randn(n, c, generator=g, device="cuda"), torch.zeros(n, c, device="cuda")], -1)
    bcoef = bcoef.contiguous()
    P = dSa = None
    if a["P"] is not None:
        P = 1 + 0.3 * torch.randn(n, d, c, generator=g, device="cuda")
        dSa = 0.1 * torch.randn(n, d, c, generator=g, device="cuda")
    ops.norm_act_bwd_apply(dout.t, x.t, coef, bcoef, P, dSa, dx.t, c, slope)
    torch.cuda.synchronize()
    dx.check_written("norm_act_bwd_apply")
    for i in samples:
        xi, do = x.ncdhw(i), dout.ncdhw(i)
        z, m, _, ez = _act(xi, coef, i, slope)
        xhat = (xi - _bc(coef[..., 2], i)) * _bc(coef[..., 3], i)
        pre = do * _bdc(P, i) + _bdc(dSa, i) if P is not None else do
        dz = pre * m
        c1, c2, c3 = (_bc(bcoef[..., k], i) for k in range(3))
        ref = c1 * (dz - c2 - xhat * c3)
        mag = dz.abs() + c2.abs() + (xhat * c3).abs() + (do * (_bdc(P, i) if P is not None else 1)).abs()
        extra = 8 * U * c1.abs() * mag + 2 * U * ref.abs()
        tile_check("norm_act_bwd_apply", dx.ncdhw(i), ref, extra, i)


def replay_maxpool_bwd_add_argmax(a, samples):
    """dskip = (accumulate ? dskip : 0) + dpool scattered to the window corner of its code: the fp32 sum of two bf16 values
    rounded once, so bit-exact."""
    from spff_b200 import ops
    g = _gen(21)
    dpool = PM.of(a["dpool"]).fill(g)
    dskip = PM.of(a["dskip"])
    acc = a["accumulate"]
    c = a["c"]
    if acc:
        dskip.fill(g)
    before = [dskip.t[i].clone() for i in samples]
    codes = torch.randint(0, 4, a["pool_argmax"][1], generator=g, device="cuda", dtype=torch.uint8)
    ops.maxpool_bwd_add_argmax(dpool.t, codes, dskip.t, c, acc)
    torch.cuda.synchronize()
    dskip.check_written("maxpool_bwd_add_argmax")
    d, h2, w2 = codes.shape[1:4]
    for i, b0 in zip(samples, before):
        onehot = F.one_hot(codes[i].long(), 4).float()                  # [d, h2, w2, c, 4]
        sc = (onehot * dpool.t[i].float().unsqueeze(-1)).view(d, h2, w2, c, 2, 2)
        sc = sc.permute(0, 1, 4, 2, 5, 3).reshape(d, 2 * h2, 2 * w2, c)
        ref = (b0.float() + sc) if acc else sc
        got = dskip.t[i]
        assert torch.equal(got, ref.to(torch.bfloat16)), f"maxpool_bwd_add_argmax: sample {i}"
        tile_check("maxpool_bwd_add_argmax", got.float().permute(3, 0, 1, 2)[None], ref.permute(3, 0, 1, 2)[None], 0.0, i)


def _convt_weight(cin, cout, g):
    return torch.randn(cin, cout, 1, 2, 2, generator=g, device="cuda") / math.sqrt(cin)


def replay_convt_k122_fwd(a, samples):
    """ConvTranspose3d (1,2,2) forward into the up half of a concat buffer against F.conv_transpose3d in fp64 on the bf16
    weight; accumulation term gamma(cin + 1) * (|x| convT |w| + |b|)."""
    from spff_b200 import ops
    g = _gen(22)
    cin, cout = a["cin"], a["cout"]
    x = PM.of(a["x"]).fill(g)
    y = PM.of(a["y"])
    wt = _convt_weight(cin, cout, g)
    b = 0.1 * torch.randn(cout, generator=g, device="cuda")
    wf, _ = ops.pack_convt_weight(wt)
    ops.convt_k122_fwd(x.t, cin, wf, b, y.t, cout)
    torch.cuda.synchronize()
    y.check_written("convt_k122_fwd")
    wq, b64 = wt.to(torch.bfloat16).double(), b.double()
    for i in samples:
        xi = x.ncdhw(i, torch.float64)
        ref = F.conv_transpose3d(xi, wq, b64, stride=(1, 2, 2)).float()
        absr = F.conv_transpose3d(xi.abs(), wq.abs(), b64.abs(), stride=(1, 2, 2))
        tile_check("convt_k122_fwd", y.ncdhw(i), ref, (gamma(cin + 1) * absr).float(), i)
        assert rel(y.ncdhw(i), ref) < 5e-3


def replay_convt_k122_dgrad(a, samples):
    """Its input gradient (out of the up half of the concat gradient) against F.conv3d with stride (1,2,2) in fp64;
    accumulation term gamma(4 cout) * (|dy| conv |w|)."""
    from spff_b200 import ops
    g = _gen(23)
    cin, cout = a["cin"], a["cout"]
    dy = PM.of(a["dy"]).fill(g)
    dx = PM.of(a["dx"])
    wt = _convt_weight(cin, cout, g)
    _, wd = ops.pack_convt_weight(wt)
    ops.convt_k122_dgrad(dy.t, cout, wd, dx.t, cin)
    torch.cuda.synchronize()
    dx.check_written("convt_k122_dgrad")
    wq = wt.to(torch.bfloat16).double()
    for i in samples:
        dyi = dy.ncdhw(i, torch.float64)
        ref = F.conv3d(dyi, wq, stride=(1, 2, 2)).float()
        absr = F.conv3d(dyi.abs(), wq.abs(), stride=(1, 2, 2))
        tile_check("convt_k122_dgrad", dx.ncdhw(i), ref, (gamma(4 * cout) * absr).float(), i)
        assert rel(dx.ncdhw(i), ref) < 5e-3


def replay_convt_k122_wgrad(a, samples):
    """dw[cin, cout, 1, 2, 2] = beta*dw0 + gradient: autograd of F.conv_transpose3d in fp64 per sample, summed; bound as
    for conv3d_k3_wgrad with N = the coarse positions."""
    from spff_b200 import ops
    g = _gen(24)
    cin, cout, beta = a["cin"], a["cout"], a["beta"]
    x = PM.of(a["x"]).fill(g)
    dy = PM.of(a["dy"]).fill(g)
    dw0 = torch.randn(a["dw"][1], generator=g, device="cuda")
    dw = dw0.clone()
    ops.convt_k122_wgrad(x.t, cin, dy.t, cout, dw, beta)
    torch.cuda.synchronize()
    ref = beta * dw0.double()
    absr = torch.zeros_like(ref)
    for i in range(x.t.shape[0]):
        for sign, acc in ((False, ref), (True, absr)):
            xi, dyi = x.ncdhw(i, torch.float64), dy.ncdhw(i, torch.float64)
            if sign:
                xi, dyi = xi.abs(), dyi.abs()
            wq = torch.zeros(dw.shape, dtype=torch.float64, device="cuda", requires_grad=True)
            F.conv_transpose3d(xi, wq, None, stride=(1, 2, 2)).backward(dyi)
            acc += wq.grad
    n, d, h, w, _ = x.t.shape
    elem_check("convt_k122_wgrad", dw, ref, sum_bound(absr, n * d * h * w) + 2 * U * beta * dw0.abs().double() + 1e-30)
    r = rel(dw - beta * dw0, ref - beta * dw0.double())
    print(f"convt_k122_wgrad {n}x{d}x{h}x{w} {cin}->{cout}: rel-L2 {r:.2e}")
    assert r < sum_rel_bound(n * d * h * w), r


def near_ties(logits):
    """test_eval_gpu.py: the two largest logits within 1e-5 (relative, floor 1) may take either arg-max."""
    top = logits.topk(2, dim=1).values
    return (top[:, 0] - top[:, 1]) <= 1e-5 * top[:, 0].abs().clamp(min=1.0)


def _head_ref(xi, w, b):
    """fp32 logits (TF32 off), and the bound of the kernel's logits: W split into bf16 hi + lo (2^-16 relative) and fp32
    accumulation of 32 products, <= 2^-15 * max_k sum|x w_k| per voxel; a softmax probability moves by at most twice
    that, plus 2^-20 for exp and the division."""
    k = w.shape[0]
    W = w.reshape(k, 32)
    torch.backends.cudnn.allow_tf32 = False
    lg = F.conv3d(xi, W.view(k, 32, 1, 1, 1), b)
    M = F.conv3d(xi.abs(), W.abs().view(k, 32, 1, 1, 1)).amax(1)          # [1, d, h, w]
    return lg, 2.0 ** -14 * M + 2.0 ** -20


def _head_common(entry, a, samples, x, w, b, labels, out):
    """Shared tally reference of head_loss_fused / head_eval: nll sum, count, confusion (near ties may move), and for
    the per-sample rows and labels_out the same per sample."""
    acc, cnt, conf = out["acc"], out["counts"], out["confusion"]
    ign = a["ignore_index"]
    n = x.t.shape[0]
    nll = nllb = 0.0
    count = ties = 0
    confr = torch.zeros(K * K, dtype=torch.int64, device="cuda")
    rows = []
    for i in range(n):
        xi = x.ncdhw(i)
        lg, dp = _head_ref(xi, w, b)
        li = labels[i:i + 1].long()
        valid = li != ign
        lse = lg.logsumexp(1)
        picked = lg.gather(1, li.clamp(max=K - 1).unsqueeze(1))[:, 0]
        s_nll = float((lse - picked)[valid].double().sum())
        nll += s_nll
        nllb += float(dp[valid].double().sum()) + sum_bound(s_nll, int(valid.sum()))
        am = lg.argmax(1)
        tie = near_ties(lg)
        ties += int((tie & valid).sum())
        ci = torch.bincount((li * K + am)[valid], minlength=K * K)
        confr += ci
        count += int(valid.sum())
        rows.append((s_nll, int(valid.sum()), ci.view(K, K), int((tie & valid).sum())))
        if out.get("labels_out") is not None and i in samples:
            got = out["labels_out"][i:i + 1].long()
            assert bool((got == am)[~tie].all()), f"{entry}: labels_out of sample {i}"
        yield i, xi, lg, dp, li, valid
    assert int(cnt) == count, f"{entry}: count {int(cnt)} != {count}"
    assert abs(float(acc) - nll) <= nllb + 1e-12 * abs(nll), f"{entry}: nll {float(acc)} vs {nll} (bound {nllb})"
    confr = confr.view(K, K)
    assert torch.equal(conf.sum(1), confr.sum(1)), f"{entry}: confusion row sums (per-label counts)"
    assert int((conf - confr).abs().sum()) <= 2 * ties, f"{entry}: confusion moved by more than the {ties} near ties"
    if out.get("sample_counts") is not None:
        for i, (s_nll, s_cnt, ci, s_ties) in enumerate(rows):
            assert int(out["sample_counts"][i]) == s_cnt
            assert int((out["sample_confusion"][i] - ci).abs().sum()) <= 2 * s_ties
            assert abs(float(out["sample_acc"][i]) - s_nll) <= nllb + 1e-12 * abs(s_nll)
    if out.get("labels_out") is not None:
        lo = out["labels_out"].long()
        lab = labels.long()
        ok = (lab != ign) & (lab < K)
        tallied = torch.bincount((lab * K + lo)[ok], minlength=K * K).view(K, K)
        assert torch.equal(tallied, conf), f"{entry}: the confusion is not the tally of labels_out"


def replay_head_loss_fused(a, samples):
    """Fused training head against F.conv3d -> cross entropy (sum / n_valid * gscale) -> autograd formulas: nll sum,
    count and confusion as in _head_common; dx per tile with the logits bound of _head_ref carried through w plus
    fp32 accumulation of 13 products. dw, db element by element: the softmax bound of _head_ref times |x| (1 for db),
    summed over the valid voxels (the hi + lo rounding of W is the same at every voxel, so it is summed, not pooled),
    plus fp32 summation of the exact terms, plus the rounding of beta * dw0."""
    from spff_b200 import ops
    g = _gen(25)
    x = PM.of(a["x"]).fill(g)
    k = a["w"][1][0]
    w = torch.randn(a["w"][1], generator=g, device="cuda") * 0.5
    b = torch.randn(k, generator=g, device="cuda") * 0.1
    labels = _labels(a["labels"], g, a["ignore_index"])
    nv = 3.0
    n_valid = torch.tensor([int(nv)], dtype=torch.int64, device="cuda")
    gs = 0.5 if a["gscale"] is not None else 1.0
    gscale = torch.tensor([gs], device="cuda") if a["gscale"] is not None else None
    out = {"acc": torch.zeros(1, dtype=torch.float64, device="cuda"), "counts": torch.zeros(1, dtype=torch.int64, device="cuda"),
           "confusion": torch.zeros(k, k, dtype=torch.int64, device="cuda")}
    dx = PM.of(a["dx"]) if a["dx"] is not None else None
    dw0 = torch.randn(a["dw"][1], generator=g, device="cuda")
    db0 = torch.randn(k, generator=g, device="cuda")
    dw, db = dw0.clone(), db0.clone()
    beta = a["beta"]
    ops.head_loss_fused(x.t, w, b, labels, a["ignore_index"], n_valid, gscale, out["acc"], out["counts"], out["confusion"],
                        dx.t if dx else None, dw, db, beta)
    torch.cuda.synchronize()
    if dx is not None:
        dx.check_written("head_loss_fused dx")
    W = w.reshape(k, 32)
    dwr = torch.zeros(k, 32, dtype=torch.float64, device="cuda")
    dbr = torch.zeros(k, dtype=torch.float64, device="cuda")
    bdw = torch.zeros(k, 32, dtype=torch.float64, device="cuda")
    bdb = torch.zeros(k, dtype=torch.float64, device="cuda")
    adw = torch.zeros_like(bdw)
    adb = torch.zeros_like(bdb)
    for i, xi, lg, dp, li, valid in _head_common("head_loss_fused", a, samples, x, w, b, labels, out):
        p = lg.softmax(1)
        oh = F.one_hot(li.clamp(max=k - 1), k).permute(0, 4, 1, 2, 3).float()
        dl = (p - oh) * valid.unsqueeze(1) * (gs / nv)
        dwr += torch.einsum("nkdhw,ncdhw->kc", dl.double(), xi.double())
        dbr += dl.double().sum(dim=(0, 2, 3, 4))
        dpv = (dp * valid).double() * (gs / nv)                         # [1, d, h, w]
        bdw += torch.einsum("ndhw,ncdhw->c", dpv, xi.abs().double()).view(1, 32)
        bdb += dpv.sum()
        adw += torch.einsum("nkdhw,ncdhw->kc", dl.abs().double(), xi.abs().double())
        adb += dl.abs().double().sum(dim=(0, 2, 3, 4))
        if dx is not None and i in samples:
            ref = torch.einsum("nkdhw,kc->ncdhw", dl, W)
            extra = (dp * valid).unsqueeze(1) * W.abs().sum(0).view(1, 32, 1, 1, 1) * (gs / nv) \
                + 2 * gamma(k) * torch.einsum("nkdhw,kc->ncdhw", dl.abs(), W.abs())
            tile_check("head_loss_fused", dx.ncdhw(i), ref, extra, i)
    npos = labels.numel()
    elem_check("head_loss_fused dw", dw, beta * dw0.double() + dwr,
               bdw + sum_bound(adw, npos) + 2 * U * (beta * dw0.double().abs() + dwr.abs()))
    elem_check("head_loss_fused db", db, beta * db0.double() + dbr,
               bdb + sum_bound(adb, npos) + 2 * U * (beta * db0.double().abs() + dbr.abs()))


def replay_head_eval(a, samples):
    """Fused evaluation head: the tally of _head_common, per sample and labels_out when the step asks for them."""
    from spff_b200 import ops
    assert a["hist"] is None, "no histogram reference here (tests/test_curves_gpu.py checks it)"
    g = _gen(26)
    x = PM.of(a["x"]).fill(g)
    k = a["w"][1][0]
    w = torch.randn(a["w"][1], generator=g, device="cuda") * 0.5
    b = torch.randn(k, generator=g, device="cuda") * 0.1
    labels = _labels(a["labels"], g, a["ignore_index"])
    z = lambda key, dt: torch.zeros(a[key][1], dtype=dt, device="cuda") if a[key] is not None else None
    out = {"acc": z("acc", torch.float64), "counts": z("counts", torch.int64), "confusion": z("confusion", torch.int64),
           "sample_acc": z("sample_acc", torch.float64), "sample_counts": z("sample_counts", torch.int64),
           "sample_confusion": z("sample_confusion", torch.int64),
           "labels_out": torch.full(a["labels_out"][1], 77, dtype=torch.uint8, device="cuda") if a["labels_out"] else None}
    ops.head_eval(x.t, w, b, labels, a["ignore_index"], out["acc"], out["counts"], out["confusion"], out["sample_acc"],
                  out["sample_counts"], out["sample_confusion"], out["labels_out"])
    torch.cuda.synchronize()
    for _ in _head_common("head_eval", a, samples, x, w, b, labels, out):
        pass


def replay_head_argmax(a, samples):
    """Arg-max label map == argmax of the fp32 logits except at near ties."""
    from spff_b200 import ops
    g = _gen(27)
    x = PM.of(a["x"]).fill(g)
    k = a["w"][1][0]
    w = torch.randn(a["w"][1], generator=g, device="cuda") * 0.5
    b = torch.randn(k, generator=g, device="cuda") * 0.1
    lab = torch.full(a["labels"][1], 77, dtype=torch.uint8, device="cuda")
    ops.head_argmax(x.t, w, b, lab)
    torch.cuda.synchronize()
    for i in samples:
        lg, _ = _head_ref(x.ncdhw(i), w, b)
        tie = near_ties(lg)
        assert bool((lab[i:i + 1].long() == lg.argmax(1))[~tie].all()), f"head_argmax: sample {i}"


def replay_count_valid(a, samples):
    from spff_b200 import ops
    g = _gen(28)
    labels = _labels(a["labels"], g, a["ignore_index"])
    out = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    ops.count_valid(labels, a["ignore_index"], out)
    want = sum(int((li != a["ignore_index"]).sum()) for li in labels)     # per sample: no 4e9-element temporaries
    assert int(out) == want


def replay_scale_by_count(a, samples):
    """g *= factor / count: fp64 reference, two fp32 roundings."""
    from spff_b200 import ops
    g = _gen(29)
    v = torch.randn(a["g"][1], generator=g, device="cuda")
    want = v.double() * a["factor"] / 12345
    cnt = torch.tensor([12345], dtype=torch.int64, device="cuda")
    ops.scale_by_count(v, cnt, a["factor"])
    elem_check("scale_by_count", v, want, 2 * U * want.abs() + 1e-45)
    z = torch.randn(a["g"][1], generator=g, device="cuda")
    ops.scale_by_count(z, torch.zeros(1, dtype=torch.int64, device="cuda"), a["factor"])
    assert bool((z == 0).all())


def replay_loss_from_tally(a, samples):
    """nll / max(count, 1) + 0.5 * (1 - mean over classes 1..K-1 of (2tp + s) / (2tp + fp + fn + s)) in fp64."""
    from spff_b200 import ops
    g = _gen(30)
    k, smooth = a["k"], a["smooth"]
    conf = torch.randint(0, 5000, (k, k), generator=g, device="cuda")
    conf[3] = 0
    cnt = conf.sum().reshape(1)
    nll = torch.tensor([0.37 * float(cnt)], dtype=torch.float64, device="cuda")
    out = torch.full((1,), float("nan"), device="cuda")
    ops.loss_from_tally(nll, cnt, conf, k, smooth, out)
    c = conf.double()
    tp = c.diag()
    fp, fn = c.sum(0) - tp, c.sum(1) - tp
    dice = ((2 * tp + smooth) / (2 * tp + fp + fn + smooth))[1:].mean()
    want = float(nll) / float(cnt) + 0.5 * (1 - float(dice))
    assert abs(float(out) - want) <= 4 * U * abs(want)


def replay_partial_colsum(a, samples):
    """out[:cols] += column sums in double: fp64 reference, the final fp32 rounding of the sum and of the add."""
    from spff_b200 import ops
    g = _gen(31)
    m = torch.randn(a["m"][1], generator=g, device="cuda")
    rows, stride, cols = a["rows"], a["row_stride"], a["cols"]
    out0 = torch.randn(a["out"][1], generator=g, device="cuda")
    out = out0.clone()
    ops.partial_colsum(m, rows, stride, cols, out)
    flat = m.reshape(-1)[:rows * stride].view(rows, stride)[:, :cols].double()
    want = out0.double().clone()
    want[:cols] += flat.sum(0)
    b = torch.zeros_like(want)                      # columns >= cols are not touched
    b[:cols] = 2 * U * (want[:cols].abs() + flat.abs().sum(0))
    elem_check("partial_colsum", out, want, b)


CONV = ("conv3d_k3_fwd", "conv3d_k3_fwd_stats", "conv3d_k3_dgrad", "conv3d_k3_dgrad_stats")

# Every public entry point of spff_b200.ops: its replay, or why a step signature is not replayed here.
ENTRY_POINTS = {
    **{e: "conv" for e in CONV},
    "conv3d_k3_wgrad": replay_conv3d_k3_wgrad,
    "conv3d_stem_fwd_stats": replay_conv3d_stem_fwd_stats,
    "conv3d_stem_wgrad": replay_conv3d_stem_wgrad,
    "in_coeffs_from_partials": replay_in_coeffs_from_partials,
    "norm_act_apply": replay_norm_act_apply,
    "norm_act_reduce": replay_norm_act_reduce,
    "norm_act_affine_apply": replay_norm_act_affine_apply,
    "norm_act_bwd_reduce": replay_norm_act_bwd_reduce,
    "norm_act_bwd_apply": replay_norm_act_bwd_apply,
    "maxpool_bwd_add_argmax": replay_maxpool_bwd_add_argmax,
    "convt_k122_fwd": replay_convt_k122_fwd,
    "convt_k122_dgrad": replay_convt_k122_dgrad,
    "convt_k122_wgrad": replay_convt_k122_wgrad,
    "head_loss_fused": replay_head_loss_fused,
    "head_eval": replay_head_eval,
    "head_argmax": replay_head_argmax,
    "count_valid": replay_count_valid,
    "scale_by_count": replay_scale_by_count,
    "loss_from_tally": replay_loss_from_tally,
    "partial_colsum": replay_partial_colsum,
    "pack_conv3_weight": "weight re-layout of [cout, cin, 3, 3, 3]; independent of the plane size, and every conv replay "
                         "packs its weight through it",
    "pack_convt_weight": "weight re-layout; independent of the plane size, and every transposed-conv replay packs through it",
    "conv3d_k3_stat_slots": "size query; the fwd_stats / dgrad_stats replays allocate from it and check every slot",
    "conv3d_stem_stat_slots": "size query; the stem replay allocates from it and checks every slot",
    "gate_tables_fwd": "gate parameter tables [c, frames]: depend on the parameters only, not on the plane size "
                       "(test_gates_gpu.py::test_gate_tables_fwd, every frames 1..16 and c 32..512)",
    "gate_tables_bwd": "gate parameter tables: parameter-only work (test_gates_gpu.py::test_gate_tables_bwd, "
                       "test_gates_gpu.py::test_variant_configurations_through_gate_tables)",
    "gate_micro_fwd": "works on per-plane statistics [n, d, c]; h, w enter only as the count h*w "
                      "(test_gates_gpu.py::test_gate_micro_fwd, planes up to 512 x 512)",
    "gate_micro_bwd": "works on per-plane sums [n, d, c, 6]; h, w enter only as the count h*w "
                      "(test_gates_gpu.py::test_gate_micro_bwd, test_gates_gpu.py::test_variant_configurations_through_gate_tables)",
    "adam_step": "flat parameter update; independent of the slice size (test_kernels_gpu.py::test_adam)",
    "workspace": "host-side scratch allocator",
}

STEP_SHAPES = ((512, 512), (200, 136))      # native slices; a rectangle whose levels 3 and 4 do not tile by 16 x 8


def _sig(v):
    from spff_b200._lib import Shape
    if isinstance(v, torch.Tensor):
        ld = v.stride(-2) if v.dim() >= 2 else max(v.numel(), 1)
        return ("T", tuple(v.shape), str(v.dtype).replace("torch.", ""), tuple(v.stride()), v.storage_offset() % max(ld, 1))
    if isinstance(v, Shape):
        return ("S", v.n, v.d, v.h, v.w)
    if isinstance(v, (tuple, list)):
        return tuple(_sig(e) for e in v)
    if v is None or isinstance(v, (bool, int, float, str)):
        return v
    return type(v).__name__


@pytest.fixture(scope="module")
def recorded():
    """{entry point: sorted distinct signatures} of the calls SPFF-UNet and PlainCore_UNet make in fit_step
    (optimize=False), predict_labels and eval_step on one slice of each STEP_SHAPES. Only the outermost ops call is
    recorded (an entry point calling another, e.g. a workspace query, is part of the first)."""
    from oracle import spff_oracle as O
    from spff_b200 import ops
    from test_model_gpu import build, load_det
    sigs = {}
    depth = [0]

    def wrap(name, fn):
        sig = inspect.signature(fn)

        def rec(*args, **kw):
            if depth[0] == 0:
                b = sig.bind(*args, **kw)
                b.apply_defaults()
                sigs.setdefault(name, set()).add(tuple((k, _sig(v)) for k, v in b.arguments.items()))
            depth[0] += 1
            try:
                return fn(*args, **kw)
            finally:
                depth[0] -= 1
        return rec

    t0 = time.time()
    with pytest.MonkeyPatch.context() as mp:
        for name, fn in list(vars(ops).items()):
            if inspect.isfunction(fn) and fn.__module__ == ops.__name__ and not name.startswith("_"):
                mp.setattr(ops, name, wrap(name, fn))
        for variant in ("SPFF-UNet", "PlainCore_UNet"):
            lit = build(variant)
            load_det(lit, variant)
            for h, w in STEP_SHAPES:
                x, lab = O.phantom_batch(1, h, w, seed=5, ignore_frac=0.02)
                xg, lg = x.cuda(), lab.cuda()
                lit.fit_step((xg, lg), optimize=False)
                lit.model.predict_labels(xg)
                lit.eval_step((xg, lg))
            del lit
        torch.cuda.synchronize()
    torch.cuda.empty_cache()
    out = {k: sorted(v, key=repr) for k, v in sigs.items()}
    print(f"\nrecorded {sum(len(v) for v in out.values())} distinct signatures of {len(out)} entry points "
          f"in {time.time() - t0:.1f} s")
    return out


@pytest.fixture(autouse=True)
def _budget(request):
    """Per-test runtime and peak allocation (the machines are shared: every test frees what it allocated)."""
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    t0 = time.time()
    yield
    torch.cuda.synchronize()
    print(f"\n[budget] {request.node.name}: {time.time() - t0:.1f} s, peak {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")
    torch.cuda.empty_cache()


@pytest.fixture(scope="module", autouse=True)
def _report():
    yield
    if WORST:
        print("\nworst error / bound per entry point:")
        for k in sorted(WORST):
            print(f"  {k:28s} {WORST[k]:.3f}")


@pytest.fixture(params=["auto", "rows", "halo"])
def conv_kernel(request):
    """Two kernels implement forward / dgrad (flattened-row: conv3_fprop.cu, halo-tile: conv3_halo.cu; the library picks one
    per shape and channel count). Every case runs under the default choice and with either kernel forced (debug key 7;
    a forced halo kernel still needs planes that tile by 16 x 8 and falls back otherwise)."""
    from spff_b200 import _lib
    _lib.lib.spff_debug_set(7, {"auto": 0, "rows": 1, "halo": 2}[request.param])
    yield request.param
    _lib.lib.spff_debug_set(7, 0)


# --------------------------------------------------------------------------------------------------------------------
# 1 + 2: the step's signatures
# --------------------------------------------------------------------------------------------------------------------
def test_every_step_entry_point_has_a_reference_or_a_reason(recorded):
    from spff_b200 import ops
    missing = sorted(set(recorded) - set(ENTRY_POINTS))
    assert not missing, f"entry points the step calls with neither a replay nor a reason: {missing}"
    public = {n for n, f in vars(ops).items() if inspect.isfunction(f) and f.__module__ == ops.__name__ and not n.startswith("_")}
    assert set(ENTRY_POINTS) <= public, sorted(set(ENTRY_POINTS) - public)
    # the shapes this file is about were seen: level 1 at 512 x 512, level 2 at 256 x 256, and the rectangle
    planes = {(s[1][2], s[1][3]) for sig in recorded["conv3d_k3_fwd_stats"] for k, s in sig if k == "x"}
    assert {(512, 512), (256, 256), (200, 136), (25, 17)} <= planes, planes
    replayed = sum(len(v) for k, v in recorded.items() if not isinstance(ENTRY_POINTS[k], str) or k in CONV)
    print(f"\n{replayed} signatures replayed against a reference:")
    for k in sorted(recorded):
        how = "replayed" if (k in CONV or not isinstance(ENTRY_POINTS[k], str)) else "not replayed: " + ENTRY_POINTS[k]
        print(f"  {k:28s} {len(recorded[k]):3d}  {how}")


def _replay_all(recorded, entry, fn):
    sigs = recorded.get(entry)
    if not sigs:
        pytest.skip(f"the step does not call {entry}")
    for s in sigs:
        a = dict(s)
        n = next(v[1][0] for v in a.values() if isinstance(v, tuple) and v and v[0] == "T")
        fn(a, list(range(n)))


@pytest.mark.parametrize("entry", CONV)
def test_replay_conv_signatures(recorded, entry, conv_kernel):
    sigs = recorded.get(entry)
    if not sigs:
        pytest.skip(f"the step does not call {entry}")
    for s in sigs:
        a = dict(s)
        n = (a.get("x") or a.get("dy"))[1][0]
        replay_conv(entry, a, list(range(n)), conv_kernel)


@pytest.mark.parametrize("entry", sorted(k for k, v in ENTRY_POINTS.items() if callable(v)))
def test_replay_step_signatures(recorded, entry):
    _replay_all(recorded, entry, ENTRY_POINTS[entry])


def test_the_checks_fire_on_one_wrong_tile():
    """The per-tile, stray-write and zero-slot assertions fail when one element of one tile is wrong: a 512 x 512
    conv output into a concat half, checked, then corrupted three ways."""
    from spff_b200 import _lib, ops
    from spff_b200._lib import Shape
    g = _gen(40)
    x = PM(1, 5, 512, 512, 32).fill(g)
    y = PM(1, 5, 512, 512, 32, ld=64, off=32)
    wt = torch.randn(32, 32, 3, 3, 3, generator=g, device="cuda") / math.sqrt(27 * 32)
    wf, _ = ops.pack_conv3_weight(wt)
    slots = ops.conv3d_k3_stat_slots(Shape(1, 5, 512, 512))
    partial = torch.full((1, slots, 2, 32), float("nan"), device="cuda")
    _lib.lib.spff_debug_set(7, 2)
    try:
        ops.conv3d_k3_fwd_stats(x.t, 32, wf, y.t, 32, partial)
        torch.cuda.synchronize()
    finally:
        _lib.lib.spff_debug_set(7, 0)
    ref = F.conv3d(x.ncdhw(0), wt.to(torch.bfloat16).float(), padding=1)
    extra = 2 * gamma(27 * 32) * F.conv3d(x.ncdhw(0).abs(), wt.to(torch.bfloat16).float().abs(), padding=1)
    y.check_written("clean")
    tile_check("corruption check", y.ncdhw(0), ref, extra)
    _check_partials("corruption check", partial, (0, ref), extra, -(-5 * 512 * 512 // slots) + 8, True, (1, 5, 512, 512), 32)
    # one element of tile 1000 (positions 128000..128127), channel 40 - 32 = 8 of the view: off by 4 ulps of the tile
    got = y.ncdhw(0).clone()
    flat = got.permute(0, 2, 3, 4, 1).reshape(-1, 32)
    p = 1000 * 128 + 77
    tile_max = float(ref.permute(0, 2, 3, 4, 1).reshape(-1, 32)[1000 * 128:1001 * 128].abs().max())
    flat[p, 8] += 4 * 2.0 ** (math.floor(math.log2(tile_max)) - 7)
    with pytest.raises(AssertionError, match=r"tile 1000 .* channels 0\.\.31"):
        tile_check("corruption check", flat.view(1, 5, 512, 512, 32).permute(0, 4, 1, 2, 3), ref, extra)
    # a write into the half the call does not own
    y.base[0, 2, 100, 100, 3] = 0.0
    with pytest.raises(AssertionError, match="does not own"):
        y.check_written("stray")
    y.base[0, 2, 100, 100, 3] = float("nan")
    # a NaN left in the owned half
    y.t[0, 1, 1, 1, 1] = float("nan")
    with pytest.raises(AssertionError, match="did not write"):
        y.check_written("unwritten")
    # a statistics slot the halo kernel should have zeroed
    mine = (512 // 16) * (512 // 8)
    assert slots > mine
    partial[0, mine + 1, 0, 5] = 1e-30
    with pytest.raises(AssertionError, match="not zero"):
        _check_partials("corruption check", partial, (0, ref), extra, -(-5 * 512 * 512 // slots) + 8, True,
                        (1, 5, 512, 512), 32)
    WORST.pop("corruption check", None)
    WORST.pop("corruption check partials", None)


# --------------------------------------------------------------------------------------------------------------------
# 3: a level-1 sample group whose concat buffers pass 2^32 elements
# --------------------------------------------------------------------------------------------------------------------
N_BIG, D, H, W = 52, 5, 512, 512             # 52 * 5 * 512 * 512 * 64 = 4.36e9 elements in a pitch-64 buffer


def _pm(n, d, h, w, c, ld=None, off=0):
    ld = ld or c
    return ("T", (n, d, h, w, c), "bfloat16", (d * h * w * ld, h * w * ld, w * ld, ld, 1), off)


def _ts(shape, dtype="float32"):
    return ("T", tuple(shape), dtype, None, 0)


@pytest.fixture
def big():
    """Skips unless 45 GiB are free; the test keeps its peak allocation under 40 GiB and frees it at the end."""
    free, _ = torch.cuda.mem_get_info()
    if free < 45 * 2 ** 30:
        pytest.skip(f"{free / 2 ** 30:.0f} GiB free: the 2^32-element group needs 45 GiB")
    torch.cuda.empty_cache()
    yield [0, N_BIG // 2, N_BIG - 1]
    peak = torch.cuda.max_memory_allocated()
    torch.cuda.empty_cache()
    assert peak < 40 * 2 ** 30, f"peak allocation {peak / 2 ** 30:.1f} GiB"


def test_large_group_numel_passes_2_to_32():
    assert N_BIG * D * H * W * 64 > 2 ** 32 and N_BIG * D * H * W * 32 > 2 ** 31


@pytest.mark.parametrize("cin,xoff,xld", [(64, 0, 64), (32, 32, 64)])
def test_large_group_conv_fwd_stats(big, cin, xoff, xld):
    """64 -> 32 reading the whole concat buffer, 32 -> 32 reading its skip half and writing into an up half."""
    a = {"x": _pm(N_BIG, D, H, W, cin, xld, xoff), "cin": cin, "cout": 32,
         "y": _pm(N_BIG, D, H, W, 32, 64 if cin == 32 else 32, 0),
         "partial": _ts((N_BIG, _slots(), 2, 32))}
    replay_conv("conv3d_k3_fwd_stats", a, big, "auto")


def _slots():
    from spff_b200 import ops
    from spff_b200._lib import Shape
    return ops.conv3d_k3_stat_slots(Shape(N_BIG, D, H, W))


def test_large_group_conv_dgrad_stats(big):
    """dec1's conv1 input gradient: 32 -> 64 channels into the whole concat gradient buffer, with its column statistics."""
    a = {"dy": _pm(N_BIG, D, H, W, 32), "cout": 32, "dx": _pm(N_BIG, D, H, W, 64), "cin": 64,
         "partial": _ts((N_BIG, _slots(), 2, 64))}
    replay_conv("conv3d_k3_dgrad_stats", a, big, "auto")


@pytest.mark.parametrize("cin,xoff", [(64, 0), (32, 32)])
def test_large_group_conv_wgrad(big, cin, xoff):
    a = {"x": _pm(N_BIG, D, H, W, cin, 64, xoff), "cin": cin, "dy": _pm(N_BIG, D, H, W, 32), "cout": 32, "beta": 1.0}
    replay_conv3d_k3_wgrad(a, big)


def test_large_group_stem(big):
    """Stem forward with statistics and its weight gradient, with y / dy in a concat half so that offsets pass 2^32."""
    replay_conv3d_stem_fwd_stats({"x": _ts((N_BIG, 1, D, H, W)), "w": _ts((32, 1, 3, 3, 3)), "cout": 32,
                                  "y": _pm(N_BIG, D, H, W, 32, 64, 32),
                                  "partial": _ts((N_BIG, _stem_slots(), 2, 32))}, big)
    torch.cuda.empty_cache()
    replay_conv3d_stem_wgrad({"x": _ts((N_BIG, 1, D, H, W)), "dy": _pm(N_BIG, D, H, W, 32, 64, 32), "cout": 32,
                              "dw": _ts((32, 1, 3, 3, 3)), "beta": 1.0}, big)


def _stem_slots():
    from spff_b200 import ops
    from spff_b200._lib import Shape
    return ops.conv3d_stem_stat_slots(Shape(N_BIG, D, H, W))


def test_large_group_affine_apply_pool_argmax(big):
    """enc1's output into the skip half of the concat buffer, pooled with arg-max codes."""
    a = {"x": _pm(N_BIG, D, H, W, 32), "c": 32, "slope": 0.01, "P": _ts((N_BIG, D, 32)), "Q": _ts((N_BIG, D, 32)),
         "y": _pm(N_BIG, D, H, W, 32, 64, 32), "ypool": _pm(N_BIG, D, H // 2, W // 2, 32),
         "pool_argmax": _ts((N_BIG, D, H // 2, W // 2, 32), "uint8")}
    replay_norm_act_affine_apply(a, big)


def test_large_group_norm_act_backward(big):
    """enc1's norm backward reads its output gradient from the skip half of the concat gradient."""
    replay_norm_act_bwd_reduce({"dout": _pm(N_BIG, D, H, W, 32, 64, 32), "x": _pm(N_BIG, D, H, W, 32), "c": 32,
                                "slope": 0.01, "plain": False, "fixed_order": True, "S": _ts((N_BIG, D, 32)),
                                "R": _ts((N_BIG, D, 32, 6))}, big)
    torch.cuda.empty_cache()
    replay_norm_act_bwd_apply({"dout": _pm(N_BIG, D, H, W, 32, 64, 32), "x": _pm(N_BIG, D, H, W, 32), "c": 32,
                               "slope": 0.01, "P": _ts((N_BIG, D, 32)), "dSa": _ts((N_BIG, D, 32)),
                               "dx": _pm(N_BIG, D, H, W, 32)}, big)


def test_large_group_maxpool_bwd_add_argmax(big):
    a = {"dpool": _pm(N_BIG, D, H // 2, W // 2, 32), "pool_argmax": _ts((N_BIG, D, H // 2, W // 2, 32), "uint8"),
         "dskip": _pm(N_BIG, D, H, W, 32, 64, 32), "c": 32, "accumulate": True}
    replay_maxpool_bwd_add_argmax(a, big)


def test_large_group_convt(big):
    """up1: 64 channels at 256 x 256 into / out of the up half of the level-1 concat (gradient) buffer."""
    fine, coarse = _pm(N_BIG, D, H, W, 32, 64, 0), _pm(N_BIG, D, H // 2, W // 2, 64)
    replay_convt_k122_fwd({"x": coarse, "cin": 64, "y": fine, "cout": 32}, big)
    torch.cuda.empty_cache()
    replay_convt_k122_dgrad({"dy": fine, "cout": 32, "dx": coarse, "cin": 64}, big)
    torch.cuda.empty_cache()
    replay_convt_k122_wgrad({"x": coarse, "cin": 64, "dy": fine, "cout": 32, "dw": _ts((64, 32, 1, 2, 2)), "beta": 1.0},
                            big)


def test_large_group_heads(big):
    """Both fused heads reading dec1's output from a pitch-64 buffer (past 2^32 elements); the training head writes its
    input gradient into another one."""
    x = _pm(N_BIG, D, H, W, 32, 64, 32)
    common = {"x": x, "w": _ts((K, 32, 1, 1, 1)), "b": _ts((K,)), "labels": _ts((N_BIG, D, H, W), "uint8"),
              "ignore_index": IGN}
    replay_head_eval({**common, "acc": _ts((1,), "float64"), "counts": _ts((1,), "int64"),
                      "confusion": _ts((K, K), "int64"), "sample_acc": _ts((N_BIG,), "float64"),
                      "sample_counts": _ts((N_BIG,), "int64"), "sample_confusion": _ts((N_BIG, K, K), "int64"),
                      "labels_out": _ts((N_BIG, D, H, W), "uint8"), "hist": None, "sample_hist": None}, big)
    torch.cuda.empty_cache()
    replay_head_loss_fused({**common, "n_valid": _ts((1,), "int64"), "gscale": None, "dx": _pm(N_BIG, D, H, W, 32, 64, 0),
                            "dw": _ts((K, 32)), "db": _ts((K,)), "beta": 1.0}, big)


def test_large_group_count_valid(big):
    """uint8 labels of a 3300-slice batch: 4.3e9 labels, past 2^32."""
    replay_count_valid({"labels": _ts((3300, D, H, W), "uint8"), "ignore_index": IGN}, big)
