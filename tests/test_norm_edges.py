"""The GroupNorm and LayerNorm kernels against fp64 on offset and near-constant groups, where one-pass statistics cancel.

Every other norm test feeds randn-like data: each group and row has a mean close to zero next to its spread.  A one-pass variance
E[x^2] - mean^2 loses (|mean| / std)^2 of relative accuracy, and centred data never shows it.  The constructors here aim at it:

  offset groups       x = mu_g + sigma N(0, 1), one mu_g (random sign) per (b, f, group), |mu_g| / sigma up to 1000 (3000 in fp32)
  channel offsets     one channel of each group offset by 1000 sigma: a large group variance, a control that passes either way
  constant groups     sigma = 0 at mu in {0, 0.1, 5, 300}, at the library's eps values (1e-5 module / InflatedGroupNorm, 1e-6 spatial / decoder)
  near-static video   x[(b t), c, h, w] = base[c, h, w] + delta N(0, 1): the decoder's temporal GroupNorm (c / 32 channels x t frames at one
                      position) sees groups whose variance is tiny next to mean^2
  offset rows         LayerNorm rows h = mu_row + sigma N(0, 1), |mu_row| / sigma up to 1000

Bound.  An fp32 input of magnitude |mu| carries only ulp(|mu|) of absolute information, and the kernels apply the norm as
fmaf(x, a, beta - m a) with a = rstd gamma: the mean is rounded to fp32 and the subtraction happens at the input's magnitude.  So the floor of
the error of a normalised value is ulp(max |x| of its group) / sqrt(var + eps) * |gamma|, and every fp32 check is
err <= K_FLOOR * floor + BASE (1 + |ref|), the last term for the roundings of the output's own arithmetic.
bf16 checks keep the half-ulp-of-output rule of test_gpu_parity.py on bf16-rounded inputs.  Everything is compared with fp64; torch's fp32
error on the same input is printed next to ours.

The CPU tests replay the accumulation order of gn_stats_kernel (thread / PT / round layout, fp32 per thread, double from the warp sum on) and of the
decoder's gn_time_tokens_kernel in numpy float32: the one-pass arithmetic fails the bound from mean / std 100 on, the shifted arithmetic passes
it everywhere, and a shifted variant whose masked tail lanes add (0 - K)^2 fails it.  The GPU tests run every kernel that consumes the
statistics at the shapes where each launch path is chosen.
"""
import math

import numpy as np
import pytest
import torch

from tests.helpers import TOL_BF16, TOL_FP32, round_bf16

K_FLOOR = 4                 # err <= K_FLOOR * floor + base: mean rounding, the product m * a, beta - m a and the fmaf each round once
BASE = 1e-6                 # base = BASE (1 + |ref|): roundings that do not scale with the offset (rstd, the products, + beta, the shifted sums)
RATIOS = (0, 10, 100, 300, 1000)
RATIOS_F32 = RATIOS + (3000,)
CONSTANTS = (0.0, 0.1, 5.0, 300.0)
GROUPS = 32


def ulp32(a):
    """Spacing of fp32 at |a| (numpy or torch, elementwise), as float64."""
    a = np.abs(np.asarray(a, dtype=np.float64)).astype(np.float32)
    return np.spacing(a).astype(np.float64)


# ---- constructors ------------------------------------------------------------------------------------------------------------------
def offset_groups(shape, ratio, seed, sigma=1.0):
    """x [B, C, F, H, W] fp32 = mu_g + sigma N(0, 1), mu_g = +-ratio * sigma * U(0.8, 1.2) per (b, f, group)."""
    B, C, F, H, W = shape
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(shape, generator=g, dtype=torch.float64) * sigma
    sign = torch.where(torch.rand(B, 1, F, GROUPS, generator=g) < 0.5, -1.0, 1.0).double()
    mu = sign * ratio * sigma * (0.8 + 0.4 * torch.rand(B, 1, F, GROUPS, generator=g, dtype=torch.float64))
    mu = mu.repeat_interleave(C // GROUPS, dim=3).permute(0, 3, 2, 1).unsqueeze(-1)           # [B, C, F, 1, 1]
    return (z + mu).float()


def channel_offset_groups(shape, seed, offset=1000.0):
    """randn with the first channel of every group offset by `offset`: the group variance is ~offset^2 / cpg, well conditioned."""
    B, C, F, H, W = shape
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(shape, generator=g, dtype=torch.float64)
    x[:, ::C // GROUPS] += offset
    return x.float()


def constant_groups(shape, mu, seed):
    """sigma = 0: every element of a group equals +-mu (sign per (b, f, group))."""
    B, C, F, H, W = shape
    g = torch.Generator().manual_seed(seed)
    sign = torch.where(torch.rand(B, 1, F, GROUPS, generator=g) < 0.5, -1.0, 1.0).double()
    v = (sign * mu).repeat_interleave(C // GROUPS, dim=3).permute(0, 3, 2, 1).unsqueeze(-1)
    return v.expand(shape).float().contiguous()


def near_static_video(b, t, C, side, delta, seed, bf16=False):
    """x [(b t), c, h, w] = base[c, h, w] + delta N(0, 1)[t, c, h, w], base ~ 4 N(0, 1).  bf16: frames differ from base by a few bf16 ulps."""
    g = torch.Generator().manual_seed(seed)
    base = 4.0 * torch.randn(b, 1, C, side, side, generator=g, dtype=torch.float64)
    noise = torch.randn(b, t, C, side, side, generator=g, dtype=torch.float64)
    if bf16:
        bb = round_bf16(base.float()).double()
        ulp = torch.exp2(torch.floor(torch.log2(bb.abs().clamp_min(1e-3))) - 7)
        x = bb + ulp * torch.round(2 * noise).clamp(-3, 3)
        return round_bf16(x.float()).reshape(b * t, C, side, side)
    return (base + delta * noise).float().reshape(b * t, C, side, side)


def offset_rows(N, C, ratio, seed):
    g = torch.Generator().manual_seed(seed)
    sign = torch.where(torch.rand(N, 1, generator=g) < 0.5, -1.0, 1.0).double()
    return (sign * ratio + torch.randn(N, C, generator=g, dtype=torch.float64)).float()


def affine(C, seed):
    g = torch.Generator().manual_seed(seed)
    return 1 + 0.2 * torch.randn(C, generator=g), 0.2 * torch.randn(C, generator=g)


# ---- fp64 references and the floor -------------------------------------------------------------------------------------------------
def _groups(x):
    """[B, C, F, H, W] -> float64 [B, F, 32, cpg * P]."""
    B, C, F, H, W = x.shape
    return x.double().permute(0, 2, 1, 3, 4).reshape(B, F, GROUPS, -1)


def group_stats64(x):
    gx = _groups(x)
    return gx.mean(-1), gx.var(-1, unbiased=False), gx.abs().amax(-1)


def _per_channel(v, C):
    """[B, F, 32] -> [B, C, F, 1, 1]"""
    return v.repeat_interleave(C // GROUPS, dim=2).permute(0, 2, 1).unsqueeze(-1).unsqueeze(-1)


def groupnorm64(x, w, b, eps):
    C = x.shape[1]
    m, v, _ = group_stats64(x)
    n = (x.double() - _per_channel(m, C)) / torch.sqrt(_per_channel(v, C) + eps)
    return n * w.double().view(1, C, 1, 1, 1) + b.double().view(1, C, 1, 1, 1)


def groupnorm_floor(x, w, eps):
    """Per element: ulp(max |x| of the group) / sqrt(var + eps) * |gamma_c|."""
    C = x.shape[1]
    _, v, amax = group_stats64(x)
    f = torch.from_numpy(ulp32(amax.numpy())) / torch.sqrt(v + eps)
    return _per_channel(f, C) * w.double().abs().view(1, C, 1, 1, 1)


def check_fp32(got, ref, floor, what):
    """err <= K_FLOOR * floor + BASE (1 + |ref|) elementwise; returns the max err."""
    err = (got.double().cpu() - ref).abs()
    ratio = (err / (K_FLOOR * floor + BASE * (1 + ref.abs()))).max().item()
    assert math.isfinite(ratio) and ratio <= 1.0, f"{what}: max err {err.max().item():.3e}, worst err / bound {ratio:.2f}"
    return err.max().item()


def check_bf16(got, ref, what, floor=None):
    """Half an ulp of the bf16 output (2^-8 |ref|, 1 % slack) + a small absolute term for outputs near zero.  `floor`: the kernel computes
    in fp32 before it rounds to bf16, so the fp32 bound of check_fp32 is added (it matters near zero and for fp32 inputs / large offsets)."""
    err = (got.double().cpu() - ref).abs()
    bound = 2 ** -8 * 1.01 * ref.abs() + 2 ** -8 * 1e-2
    if floor is not None:
        bound = bound + K_FLOOR * floor + BASE * (1 + ref.abs())
    ratio = (err / bound).max().item()
    assert math.isfinite(ratio) and ratio <= 1.0, f"{what}: max err {err.max().item():.3e}, worst err / bound {ratio:.2f}"
    return err.max().item()


# ---- CPU: float32 replays of the kernels' accumulation order -----------------------------------------------------------------------
F32 = np.float32


def gn_plan(cpg, P):
    """neurons_b200/csrc/norm_kernels.cu gn_plan."""
    total = cpg * P
    cap = 512 * 16 * 8
    splits = -(-total // cap)
    per = -(-total // splits)
    best, th, pt = -1, 512, 16
    for t in (64, 128, 256, 512):
        for q in (4, 5, 8, 10, 16):
            chunk = t * q * 8
            if chunk >= per and (best < 0 or chunk < best or (chunk == best and t > th)):
                best, th, pt = chunk, t, q
    return th, pt, splits


def _fma32(a, b, c):
    return (a.astype(np.float64) * b + c).astype(F32)


def _warp_sum32(v):
    """Butterfly of warp_sum over [TH] lanes (32-lane warps), fp32; lane 0 of each warp -> [TH / 32]."""
    w = v.reshape(-1, 32).copy()
    for o in (16, 8, 4, 2, 1):
        w = (w + w[:, np.arange(32) ^ o]).astype(F32)
    return w[:, 0]


def shift_of(xg):
    """gn_stats_kernel's K for fp32 input: the fp32 mean of the first min(P, 8) elements of the group's first channel, summed in order."""
    v = np.ascontiguousarray(xg, dtype=F32).reshape(-1)[:min(xg.shape[1], 8)]
    acc = F32(0)
    for t in v:
        acc = F32(acc + t)
    return F32(acc / F32(v.size))


def _warp_sum64(v):
    """The same butterfly in double."""
    w = v.reshape(-1, 32).copy()
    for o in (16, 8, 4, 2, 1):
        w = w + w[:, np.arange(32) ^ o]
    return w[:, 0]


def emulate_gn_stats(xg, bf16=False, vec=True, shifted=True, tail_mutant=False):
    """gn_stats_kernel on one group: xg float32 [cpg, P] (bf16-representable when bf16).  Returns (sum, sum of squares) in double,
    summed over splits as gn_finalize_one does.  fp32 input accumulates x - K (K = shift_of), bf16 input x itself; each thread's sums are
    un-shifted in double before the warp sum.  shifted=False: one-pass fp32 sums of x and x^2 per thread AND per warp (the warp sum in
    fp32), the arithmetic the kernel had before."""
    cpg, P = xg.shape
    flat = np.ascontiguousarray(xg, dtype=F32).reshape(-1)
    total = flat.size
    th, pt, splits = gn_plan(cpg, P)
    chunk = th * pt * 8
    K = shift_of(xg) if shifted and not bf16 else F32(0)
    a = c2 = 0.0
    for sp in range(splits):
        e0 = sp * chunk
        s = np.zeros(th, F32)
        ss = np.zeros(th, F32)
        n = np.zeros(th, np.int64)
        tid = np.arange(th)
        if vec:
            # packed fp32x2 accumulators: lane 0 takes the even elements of each vector, lane 1 the odd ones; added at the end
            s2 = np.zeros((th, 2), F32)
            ss2 = np.zeros((th, 2), F32)
            V = 8 if bf16 else 4
            for rd in range(8 // V):
                base_e = e0 + rd * th * pt * V
                for i in range(pt):
                    e = base_e + (i * th + tid) * V
                    ok = e < total
                    vals = np.where(ok[:, None], flat[np.minimum(e, total - V)[:, None] + np.arange(V)], F32(0)).astype(F32)
                    d = (vals - K).astype(F32)
                    okv = np.ones_like(ok) if tail_mutant else ok    # mutant: masked lanes add (0 - K), (0 - K)^2; n counts valid ones
                    for j in range(0, V, 2):
                        pair = d[:, j:j + 2]
                        s2 = np.where(okv[:, None], (s2 + pair).astype(F32), s2)
                        ss2 = np.where(okv[:, None], _fma32(pair, pair, ss2), ss2)
                    n += np.where(ok, V, 0)
            s = (s2[:, 0] + s2[:, 1]).astype(F32)
            ss = (ss2[:, 0] + ss2[:, 1]).astype(F32)
        else:
            e1 = min(total, e0 + chunk)
            for e in range(e0, e1, th):
                idx = e + tid
                ok = idx < e1
                d = (flat[np.minimum(idx, total - 1)] - K).astype(F32)
                s = np.where(ok, (s + d).astype(F32), s)
                ss = np.where(ok, _fma32(d, d, ss), ss)
                n += ok
        if shifted:                                       # each thread un-shifts in double, the warp sums in double
            dk, sd, ssd = float(K), s.astype(np.float64), ss.astype(np.float64)
            ws, wss = _warp_sum64(n * dk + sd), _warp_sum64(n * dk * dk + (2 * dk * sd + ssd))
        else:
            ws, wss = _warp_sum32(s).astype(np.float64), _warp_sum32(ss).astype(np.float64)
        for i in range(ws.size):
            a += ws[i]
            c2 += wss[i]
    return a, c2


def emulate_gn_apply(xg, sums, gamma, beta, eps):
    """gn_finalize_one + the kernels' fmaf(x, a, beta - m a) on one group; xg [cpg, P], gamma / beta [cpg]."""
    a, c2 = sums
    cnt = xg.size
    m = a / cnt
    var = max(c2 / cnt - m * m, 0.0)
    mean, rstd = F32(m), F32(1.0 / math.sqrt(var + eps))
    sa = (rstd * gamma.astype(F32)).astype(F32)
    sb = (beta.astype(F32) - (mean * sa).astype(F32)).astype(F32)
    return _fma32(xg.astype(F32), sa[:, None], sb[:, None])


def _group_case(ratio, cpg, P, seed, bf16=False, sigma=1.0):
    rng = np.random.default_rng(seed)
    mu = (1 if rng.random() < 0.5 else -1) * ratio * sigma
    x = (mu + sigma * rng.standard_normal((cpg, P))).astype(F32)
    if bf16:
        x = round_bf16(torch.from_numpy(x)).numpy()
    gamma = (1 + 0.2 * rng.standard_normal(cpg)).astype(F32)
    beta = (0.2 * rng.standard_normal(cpg)).astype(F32)
    return x, gamma, beta


def _emulated_err_over_bound(x, gamma, beta, eps, **kw):
    out = emulate_gn_apply(x, emulate_gn_stats(x, **kw), gamma, beta, eps).astype(np.float64)
    xd = x.astype(np.float64)
    m, v = xd.mean(), xd.var()
    ref = (xd - m) / math.sqrt(v + eps) * gamma.astype(np.float64)[:, None] + beta.astype(np.float64)[:, None]
    floor = ulp32(np.abs(xd).max()) / math.sqrt(v + eps) * np.abs(gamma.astype(np.float64))[:, None]
    return (np.abs(out - ref) / (K_FLOOR * floor + BASE * (1 + np.abs(ref)))).max()


# (cpg, P, vec, bf16): one group of the 64 x 64 level (10 x 4096, one CTA of 512 x 10), two splits (20 x 4096), a partial last chunk
# (10 x 64 in a 64 x 4 x 8 chunk), the element loop (3 x 15) and bf16 vectors
EMU_SHAPES = [(10, 4096, True, False), (20, 4096, True, False), (10, 64, True, False), (3, 15, False, False), (10, 4096, True, True),
              (20, 4096, True, True)]


@pytest.mark.parametrize("cpg,P,vec,bf16", EMU_SHAPES)
@pytest.mark.parametrize("ratio", RATIOS_F32)
def test_emulated_shifted_gn_stats_meet_the_bound(cpg, P, vec, bf16, ratio):
    if bf16 and ratio > 30:
        pytest.skip("bf16 carries 8 bits: offsets beyond ~30 sigma are not a bf16 group with a spread")
    x, gamma, beta = _group_case(ratio, cpg, P, seed=ratio + cpg + P, bf16=bf16)
    r = _emulated_err_over_bound(x, gamma, beta, 1e-5, vec=vec, bf16=bf16)
    assert r <= 1.0, r


@pytest.mark.parametrize("cpg,P,vec", [(10, 4096, True), (20, 4096, True), (3, 15, False)])
@pytest.mark.parametrize("ratio", [100, 300, 1000, 3000])
def test_emulated_one_pass_gn_stats_fail_the_bound(cpg, P, vec, ratio):
    """The arithmetic before the shift (fp32 sums of x and x^2 per thread and warp) is caught from mean / std 100 on (worst of four
    groups: at 100 the one-pass error is about the bound, so a single group may land below it)."""
    r = max(_emulated_err_over_bound(*_group_case(ratio, cpg, P, seed=ratio + cpg + P + i), 1e-5, vec=vec, shifted=False) for i in range(4))
    assert r > 1.0, r


@pytest.mark.parametrize("mu", CONSTANTS)
@pytest.mark.parametrize("eps", [1e-5, 1e-6])
def test_emulated_shifted_gn_stats_on_constant_groups(mu, eps):
    x = np.full((10, 4096), mu, F32)
    gamma, beta = np.full(10, 1.1, F32), np.full(10, 0.1, F32)
    assert _emulated_err_over_bound(x, gamma, beta, eps) <= 1.0


def test_emulated_tail_lanes_must_be_masked():
    """With the shift, a lane past the end of the group that adds its zero vector contributes (0 - K) and (0 - K)^2: caught."""
    x, gamma, beta = _group_case(300, 10, 64, seed=3)
    assert _emulated_err_over_bound(x, gamma, beta, 1e-5) <= 1.0
    assert _emulated_err_over_bound(x, gamma, beta, 1e-5, tail_mutant=True) > 1.0


def emulate_decoder_gn(vals, gamma, beta, eps, shifted=True):
    """gn_time_tokens_kernel for one (b, position, group): vals float32 [t, cpg] (frame-major, the kernel's loop order)."""
    v = vals.astype(F32)
    K = v[0, 0] if shifted else F32(0)
    s = ss = F32(0)
    for f in range(v.shape[0]):
        for j in range(v.shape[1]):
            d = F32(v[f, j] - K)
            s = F32(s + d)
            ss = F32(np.float64(d) * d + ss)
    n = F32(v.size)
    mean = F32(s / n)
    var = max(F32(np.float64(-mean) * mean + F32(ss / n)), F32(0))
    rstd = F32(1.0 / math.sqrt(float(F32(var + F32(eps)))))
    if shifted:
        c = ((v - K).astype(F32) - mean).astype(F32)
    else:
        c = (v - mean).astype(F32)
    return ((c * rstd).astype(F32) * gamma[None, :] + beta[None, :]).astype(F32)


@pytest.mark.parametrize("cpg", [1, 2, 4])
@pytest.mark.parametrize("mean,std", [(5.0, 0.1), (5.0, 0.01), (50.0, 0.1), (4.0, 1e-3), (0.0, 1.0)])
def test_emulated_decoder_gn(cpg, mean, std):
    rng = np.random.default_rng(cpg)
    worst = {True: 0.0, False: 0.0}
    eps = 1e-6
    for _ in range(200):
        vals = (mean + std * rng.standard_normal((6, cpg))).astype(F32)
        gamma = (1 + 0.2 * rng.standard_normal(cpg)).astype(F32)
        beta = (0.2 * rng.standard_normal(cpg)).astype(F32)
        vd = vals.astype(np.float64)
        ref = (vd - vd.mean()) / math.sqrt(vd.var() + eps) * gamma + beta
        floor = ulp32(np.abs(vd).max()) / math.sqrt(vd.var() + eps) * np.abs(gamma.astype(np.float64))
        for sh in (True, False):
            out = emulate_decoder_gn(vals, gamma, beta, eps, shifted=sh)
            worst[sh] = max(worst[sh], (np.abs(out - ref) / (K_FLOOR * floor + BASE * (1 + np.abs(ref)))).max())
    assert worst[True] <= 1.0, worst
    if mean / std >= 50:
        assert worst[False] > 1.0, worst          # the one-pass fp32 arithmetic fails on near-static groups


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
DEV = "cuda"
GN_EPS_MODULE = 1e-6        # the motion module's GroupNorm (ops.GN_EPS), the spatial transformer's and the decoder's
GN_EPS_RESNET = 1e-5        # InflatedGroupNorm of ResnetBlock3D


def _to_layout(x, layout):
    """Same logical [B, C, F, H, W] tensor over [B, C, F, H, W] ("bcfhw") or [B, F, C, H, W] ("bfchw") storage."""
    return x.contiguous() if layout == "bcfhw" else x.permute(0, 2, 1, 3, 4).contiguous().permute(0, 2, 1, 3, 4)


def _gn_cfg(C):
    import neurons_b200 as nb
    return nb.ModuleConfig(C, heads=1, pos_enc=False)


def _torch_gn_err(x, w, b, eps, ref):
    """torch fp32 group_norm's error on the same input, printed next to ours."""
    B, C, F, H, W = x.shape
    t = torch.nn.functional.group_norm(x.float().permute(0, 2, 1, 3, 4).reshape(B * F, C, H, W), GROUPS, w, b, eps)
    return (t.reshape(B, F, C, H, W).permute(0, 2, 1, 3, 4).double() - ref).abs().max().item()


def _check_stats(mean, rstd, x, eps, what):
    """mean: |m - m64| <= ulp(m64) + 1e-6 sigma (the fp32 rounding of the mean, the shifted sums); rstd: relative 5e-6 against fp64."""
    m64, v64, _ = group_stats64(x)
    m64, v64 = m64.reshape(-1, GROUPS), v64.reshape(-1, GROUPS)
    r64 = 1 / torch.sqrt(v64 + eps)
    em = (mean.double().cpu() - m64).abs()
    bm = torch.from_numpy(ulp32(m64.numpy())) + 1e-6 * v64.sqrt()
    assert (em <= bm).all(), f"{what}: mean err / bound {(em / bm).max().item():.2f}"
    er = (rstd.double().cpu() / r64 - 1).abs().max().item()
    assert er <= 5e-6, f"{what}: rstd relative err {er:.2e}"


# (C, F, H, W, B): splits 1 (10 x 4096 in one CTA), 2 (C = 640 @ 64 x 64), 3 (C = 320 @ 128 x 128), a partial last chunk (C = 320 @ 8 x 8),
# cpg 3 (C = 96) and a ragged 3 x 5 latent (element loop)
GN_SHAPES = [(320, 2, 64, 64, 1), (640, 1, 64, 64, 1), (320, 1, 128, 128, 1), (320, 4, 8, 8, 2), (96, 2, 8, 8, 1), (320, 3, 3, 5, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("C,F,H,W,B", GN_SHAPES)
@pytest.mark.parametrize("layout", ["bcfhw", "bfchw"])
@pytest.mark.parametrize("ratio", RATIOS_F32)
def test_groupnorm_stats_and_sums_fp32_offset(C, F, H, W, B, layout, ratio):
    from neurons_b200 import ops
    x = offset_groups((B, C, F, H, W), ratio, seed=C + H + ratio)
    xd = _to_layout(x.to(DEV), layout)
    mean, rstd = ops.groupnorm_stats(_gn_cfg(C), xd)
    _check_stats(mean, rstd, x, GN_EPS_MODULE, f"stats ratio {ratio}")
    sums = ops.groupnorm_sums(xd).cpu()
    n = (C // GROUPS) * H * W
    m, v = sums[:, 0] / n, sums[:, 1] / n - (sums[:, 0] / n) ** 2
    m64, v64, _ = group_stats64(x)
    assert ((m - m64.reshape(-1)).abs() <= 1e-6 * v64.reshape(-1).sqrt() + 1e-12 * m64.abs().reshape(-1)).all()
    assert ((v - v64.reshape(-1)).abs() <= 1e-5 * v64.reshape(-1)).all(), (v / v64.reshape(-1) - 1).abs().max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("C,F,H,W,B", GN_SHAPES)
@pytest.mark.parametrize("layout", ["bcfhw", "bfchw"])
@pytest.mark.parametrize("ratio", RATIOS)
def test_groupnorm_stats_bf16_offset(C, F, H, W, B, layout, ratio):
    """bf16 inputs (the rounded offset groups; at 1000 sigma bf16 keeps ~2 significant bits of the spread): statistics against fp64 of the
    values the kernel reads."""
    from neurons_b200 import ops
    x = round_bf16(offset_groups((B, C, F, H, W), ratio, seed=C + H + ratio))
    xd = _to_layout(x.to(DEV, torch.bfloat16), layout)
    mean, rstd = ops.groupnorm_stats(_gn_cfg(C), xd)
    _check_stats(mean, rstd, x, GN_EPS_MODULE, f"bf16 stats ratio {ratio}")


@pytest.mark.gpu
@pytest.mark.parametrize("C,F,H,W,B", [(320, 2, 64, 64, 1), (640, 1, 64, 64, 1), (96, 2, 8, 8, 1), (320, 3, 3, 5, 2)])
@pytest.mark.parametrize("kind", ["channel", "constant"])
def test_groupnorm_stats_controls(C, F, H, W, B, kind):
    """Between-channel offsets (large variance: passes before and after the shift) and constant groups (var 0: rstd = 1 / sqrt(eps))."""
    from neurons_b200 import ops
    xs = [channel_offset_groups((B, C, F, H, W), seed=C)] if kind == "channel" else [constant_groups((B, C, F, H, W), mu, seed=C) for mu in CONSTANTS]
    for x in xs:
        mean, rstd = ops.groupnorm_stats(_gn_cfg(C), x.to(DEV))
        _check_stats(mean, rstd, x, GN_EPS_MODULE, kind)


@pytest.mark.gpu
@pytest.mark.parametrize("C,F,H,W,B", [(320, 2, 64, 64, 1), (640, 1, 64, 64, 1), (320, 4, 8, 8, 2), (96, 2, 8, 8, 1), (320, 3, 3, 5, 2)])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("ratio", RATIOS_F32)
def test_groupnorm_tokens_offset(C, F, H, W, B, dtype, ratio):
    """gn_tokens: the 64 x 64 bf16 kernel (C % 64 == 0, P % 64 == 0) and the generic bf16 / fp32 kernel."""
    from neurons_b200 import ops
    if dtype == torch.bfloat16 and ratio > 30:
        ratio = 30                               # bf16: the largest offset whose group still has a spread of a few ulps
    x = offset_groups((B, C, F, H, W), ratio, seed=C + W + ratio)
    if dtype == torch.bfloat16:
        x = round_bf16(x)
    w, b = affine(C, C)
    tok = ops.groupnorm_tokens(_gn_cfg(C), _to_layout(x.to(DEV, dtype), "bfchw"), w.to(DEV), b.to(DEV))
    ref = groupnorm64(x, w, b, GN_EPS_MODULE).permute(0, 2, 3, 4, 1).reshape(-1, C)
    if dtype == torch.float32:
        floor = groupnorm_floor(x, w, GN_EPS_MODULE).expand(x.shape).permute(0, 2, 3, 4, 1).reshape(-1, C)
        err = check_fp32(tok, ref, floor, f"tokens ratio {ratio}")
        print(f"gn_tokens fp32 C={C} ratio {ratio}: ours {err:.2e}  torch fp32 {_torch_gn_err(x, w, b, GN_EPS_MODULE, groupnorm64(x, w, b, GN_EPS_MODULE)):.2e}")
    else:
        check_bf16(tok, ref, f"bf16 tokens ratio {ratio}")


@pytest.mark.gpu
@pytest.mark.parametrize("C,F,H,W,B", [(320, 2, 64, 64, 1), (640, 4, 16, 16, 1), (320, 8, 8, 8, 1)])
@pytest.mark.parametrize("ratio", [0, 10, 30])
def test_groupnorm_linear_offset(C, F, H, W, B, ratio):
    """The GroupNorm-fused proj_in GEMM (bf16, offsets bf16 can carry) against gn_tokens + linear (same operands, same accumulation)
    and against fp64: half an ulp of the bf16 tokens, propagated through |W| (sum over k of |w_k| half-ulps), plus the fp32 accumulation."""
    from neurons_b200 import lib as nlib
    from neurons_b200 import ops
    x = round_bf16(offset_groups((B, C, F, H, W), ratio, seed=C + ratio))
    xd = _to_layout(x.to(DEV, torch.bfloat16), "bfchw")
    gw, gb = affine(C, 7)
    g = torch.Generator().manual_seed(C)
    wt = round_bf16((torch.rand(C, C, generator=g) * 2 - 1) / math.sqrt(C))
    bias = 0.1 * torch.randn(C, generator=g)
    fused = ops.groupnorm_linear(_gn_cfg(C), xd, gw.to(DEV), gb.to(DEV), wt.to(DEV, torch.bfloat16), bias.to(DEV))
    tok = ops.groupnorm_tokens(_gn_cfg(C), xd, gw.to(DEV), gb.to(DEV))
    h2 = torch.empty_like(fused)
    ops.linear(tok, wt.to(DEV, torch.bfloat16), bias.to(DEV), nlib.EPI_STORE, h=h2, want_out=False)
    assert torch.equal(fused, h2)
    n64 = groupnorm64(x, gw, gb, GN_EPS_MODULE).permute(0, 2, 3, 4, 1).reshape(-1, C)
    ref = n64 @ wt.double().T + bias.double()
    bound = (2 ** -8 * n64.abs()) @ wt.double().abs().T * 1.01 + 1e-4
    err = (fused.double().cpu() - ref).abs()
    assert (err <= bound).all(), (err / bound).max().item()


@pytest.mark.gpu
@pytest.mark.parametrize("C,F,H,W,B,layout", [(320, 2, 64, 64, 1, "bcfhw"), (640, 1, 64, 64, 1, "bfchw"), (96, 2, 8, 8, 1, "bcfhw"),
                                              (320, 3, 3, 5, 2, "bfchw")])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("eps", [GN_EPS_RESNET, GN_EPS_MODULE])
@pytest.mark.parametrize("silu", [False, True])
@pytest.mark.parametrize("stats", ["own", "sums", "fp64"])
def test_inflated_groupnorm_offset(C, F, H, W, B, layout, dtype, eps, silu, stats):
    """InflatedGroupNorm +- SiLU with its own statistics pass, with groupnorm_sums, and with fp64 sums handed in.  Offset 1000 sigma
    (fp32), 30 sigma (bf16); constant groups in both."""
    from neurons_b200 import ops
    ratios = (100, 1000, 3000) if dtype == torch.float32 else (30,)
    cases = [offset_groups((B, C, F, H, W), r, seed=C + r) for r in ratios] + [constant_groups((B, C, F, H, W), mu, seed=3) for mu in CONSTANTS]
    w, b = affine(C, 11)
    for x in cases:
        if dtype == torch.bfloat16:
            x = round_bf16(x)
        xd = _to_layout(x.to(DEV, dtype), layout)
        sums = None
        if stats == "sums":
            sums = ops.groupnorm_sums(xd)
        elif stats == "fp64":
            gx = _groups(x)
            sums = torch.stack([gx.sum(-1), (gx * gx).sum(-1)], -1).reshape(-1, 2).to(DEV)
        y = ops.inflated_groupnorm(xd, w.to(DEV), b.to(DEV), eps, silu=silu, sums=sums)
        ref = groupnorm64(x, w, b, eps)
        floor = groupnorm_floor(x, w, eps)
        if silu:
            ref = torch.nn.functional.silu(ref)           # |silu'| <= 1.1: the floor carries over (the fast silu adds ~2 ulps: in the base)
        if dtype == torch.float32:
            check_fp32(y, ref, 1.1 * floor, f"inflated gn {stats}")
        else:
            check_bf16(y, ref, f"bf16 inflated gn {stats}", 1.1 * floor)


@pytest.mark.gpu
@pytest.mark.parametrize("C", [320, 640, 1280, 96])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
@pytest.mark.parametrize("ratio", [0, 10, 100, 1000])
@pytest.mark.parametrize("with_pe", [False, True])
def test_layernorm_pe_offset_rows(C, dtype, ratio, with_pe):
    """The standalone LayerNorm(+pe) kernels (two-pass fp32): the vec kernel (C = 320 / 640 / 1280) and the generic kernel (C = 96)."""
    import neurons_b200 as nb
    from neurons_b200 import ops
    from oracle import motion_oracle as mo
    B, F, H, W = 1, 8, 8, 8
    N = B * F * H * W
    h = offset_rows(N, C, ratio, seed=C + ratio)
    w, b = affine(C, 5)
    pe = mo.positional_encoding(24, C)
    ref = torch.nn.functional.layer_norm(h.double(), (C,), w.double(), b.double(), 1e-5)
    if with_pe:
        ref = ref + pe.double()[(torch.arange(N) // (H * W)) % F]
    out = ops.layernorm_pe(nb.ModuleConfig(C), (B, F, H, W), h.to(DEV), w.to(DEV), b.to(DEV), pe.to(DEV) if with_pe else None, dtype)
    hd = h.double()
    floor = torch.from_numpy(ulp32(hd.abs().amax(1, keepdim=True).numpy())) / torch.sqrt(hd.var(1, unbiased=False, keepdim=True) + 1e-5) * w.double().abs()
    if dtype == torch.float32:
        err = check_fp32(out, ref, floor, f"layernorm ratio {ratio}")
        t = torch.nn.functional.layer_norm(h, (C,), w, b, 1e-5).double() + (ref - torch.nn.functional.layer_norm(h.double(), (C,), w.double(), b.double(), 1e-5))
        print(f"layernorm C={C} ratio {ratio}: ours {err:.2e}  torch fp32 {(t - ref).abs().max().item():.2e}")
    else:
        check_bf16(out, ref, f"bf16 layernorm ratio {ratio}", floor)


def _decoder_fp64(p, x, weight, t, cfg, dn=None):
    """oracle/decoder_oracle.py temporal_blend_reference_order in fp64 with an optional perturbation dn of the GroupNorm output."""
    bt, c, h, w = x.shape
    res = x.double().reshape(bt // t, t, c, h, w).permute(0, 3, 4, 1, 2).reshape(-1, t, c)
    n = torch.nn.functional.group_norm(res.transpose(1, 2), cfg.groups, p["group_norm.weight"], p["group_norm.bias"], cfg.eps).transpose(1, 2)
    if dn is not None:
        n = n + dn
    lin = lambda z, k: torch.nn.functional.linear(z, p[k + ".weight"], p[k + ".bias"])
    dh = c // cfg.heads
    q, k, v = (lin(n, nm).view(-1, t, cfg.heads, dh).transpose(1, 2) for nm in ("to_q", "to_k", "to_v"))
    o = torch.nn.functional.scaled_dot_product_attention(q, k, v).transpose(1, 2).reshape(-1, t, c)
    o = lin(o, "to_out.0") + res
    o = o.reshape(bt // t, h, w, t, c).permute(0, 3, 4, 1, 2).reshape(bt, c, h, w)
    return weight * x.double() + (1 - weight) * o


@pytest.mark.gpu
@pytest.mark.parametrize("C", [32, 64, 128])
@pytest.mark.parametrize("delta", [3e-2, 1e-2, 1e-3])
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16"])
def test_decoder_temporal_gn_near_static(C, delta, dtype):
    """The decoder's temporal attention on near-static frames (cpg 1 / 2 / 4), against the fp64 oracle.  fp32: the GroupNorm floor is
    propagated through the block in fp64 (the output change when every normalised value moves by its floor with a random sign, the larger
    of two draws); bound = K_FLOOR * that + TOL_FP32 for the GEMMs and the attention.  bf16: TOL_BF16 + half an ulp of the output."""
    from oracle import decoder_oracle as do
    from neurons_b200 import video_decoder as vd
    from tests.test_video_decoder import FakeAttention
    if dtype == torch.bfloat16 and delta != 1e-2:
        pytest.skip("bf16 frames are built from bf16 ulps, not delta")
    cfg = do.DecoderAttnConfig(C)
    params = do.make_params(cfg, C)
    x = near_static_video(1, 6, C, 12, delta, seed=C, bf16=dtype == torch.bfloat16)
    if dtype == torch.bfloat16:
        params = {k: round_bf16(v) for k, v in params.items()}
    p64 = {k: v.double() for k, v in params.items()}
    attn = FakeAttention(cfg, params).cuda().to(dtype).eval()
    weight = 0.0
    with torch.no_grad():
        y = vd.temporal_attention_blend(x.cuda().to(dtype), attn, torch.nn.Parameter(torch.tensor([weight])).cuda(), 6)
    ref = _decoder_fp64(p64, x, weight, 6, cfg)
    err = (y.double().cpu() - ref).abs().max().item()
    if dtype == torch.float32:
        res = x.double().reshape(1, 6, C, 12, 12).permute(0, 3, 4, 1, 2).reshape(-1, 6, C)
        gx = res.reshape(-1, 6, GROUPS, C // GROUPS)
        var = gx.var((1, 3), unbiased=False, keepdim=True)
        amax = gx.abs().amax((1, 3), keepdim=True)
        floor = (torch.from_numpy(ulp32(amax.numpy())) / torch.sqrt(var + cfg.eps)).expand(gx.shape).reshape(res.shape)
        floor = floor * p64["group_norm.weight"].abs()
        g = torch.Generator().manual_seed(1)
        prop = max((_decoder_fp64(p64, x, weight, 6, cfg, floor * (2 * torch.randint(0, 2, floor.shape, generator=g) - 1)) - ref).abs().max().item()
                   for _ in range(2))
        bound = K_FLOOR * prop + TOL_FP32
    else:
        bound = TOL_BF16 + 2 ** -8 * ref.abs().max().item()
    print(f"decoder C={C} delta {delta} {dtype}: err {err:.2e} bound {bound:.2e}")
    assert math.isfinite(err) and err <= bound, (err, bound)


def _module_case(C, F, side, B, ratio, seed, bias_offset=0.0, dtype=torch.float32):
    from oracle import motion_oracle as mo
    cfg = mo.MotionConfig(C)
    params = mo.make_params(cfg, seed)
    params["temporal_transformer.proj_in.bias"] = params["temporal_transformer.proj_in.bias"] + bias_offset
    x = offset_groups((B, C, F, side, side), ratio, seed=seed)
    if dtype == torch.bfloat16:
        params, x = {k: round_bf16(v) for k, v in params.items()}, round_bf16(x)
    x = _to_layout(x, "bfchw")
    ref = mo.forward_reference_order({k: v.double() for k, v in params.items()}, x.double(), cfg)
    return cfg, params, x, ref


@pytest.mark.gpu
@pytest.mark.parametrize("mode,C", [("fma", 640), ("x6", 640), ("x3", 320), ("x3", 640)])
def test_motion_module_offset_input(mode, C):
    """Whole fp32 module calls on x offset by 300 sigma per group (gn_stats, gn_tokens and its x3 / x6 plane writers).  The exact modes
    also get proj_in.bias + 20 (LayerNorm rows ~30 sigma off zero).  Bound: TOL_FP32 + 4 ulp of the output (y = x + ... carries |x| ~ 360)."""
    from tests import helpers
    cfg, params, x, ref = _module_case(C, 8, 8, 1, 300, seed=C, bias_offset=0.0 if mode == "x3" else 20.0)
    m = helpers.mirror_module(cfg, params, DEV)
    if mode != "x3":
        m.__dict__["_nmm_fp32_fma" if mode == "fma" else "_nmm_fp32_exact"] = True
    with torch.no_grad():
        y = m(x.to(DEV), None, None)
    err = (y.double().cpu() - ref).abs().max().item()
    bound = TOL_FP32 + 4 * ulp32(ref.abs().max().item())
    print(f"module {mode} C={C}: err {err:.2e} bound {bound:.2e}")
    assert math.isfinite(err) and err <= bound, (err, bound)


@pytest.mark.gpu
def test_fused_module_bf16_offset_input():
    """The one-kernel bf16 C = 320 module (its phase 0 finalises gn_stats' partials), x offset by 30 sigma per group."""
    from tests import helpers
    cfg, params, x, ref = _module_case(320, 8, 16, 2, 30, seed=3, dtype=torch.bfloat16)
    m = helpers.mirror_module(cfg, params, DEV, torch.bfloat16)
    with torch.no_grad():
        y = m(x.to(DEV, torch.bfloat16), None, None)
    err = (y.double().cpu() - ref).abs().max().item()
    bound = TOL_BF16 + 2 ** -8 * ref.abs().max().item()
    assert math.isfinite(err) and err <= bound, (err, bound)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["x3", "fma", "x6", "bf16"])
def test_spatial_transformer_offset_input(mode):
    """One spatial Transformer3DModel call with hidden states offset per group (300 sigma fp32, 30 sigma bf16; GroupNorm eps 1e-6)."""
    import neurons_b200 as nb
    from oracle import spatial_oracle as so
    cfg = so.SpatialConfig(320, 8, 1, 768, True)
    params = so.make_params(cfg, 4)
    _, ctx = so.make_inputs(cfg, 1, 2, 16, 16, 77, 5)
    dtype = torch.bfloat16 if mode == "bf16" else torch.float32
    x = offset_groups((1, 320, 2, 16, 16), 30 if mode == "bf16" else 300, seed=6)
    if mode == "bf16":
        params, x, ctx = {k: round_bf16(v) for k, v in params.items()}, round_bf16(x), round_bf16(ctx)
    m = nb.Transformer3DModel(num_attention_heads=8, attention_head_dim=40, in_channels=320, cross_attention_dim=768,
                              unet_use_cross_frame_attention=False, unet_use_temporal_attention=False)
    m.load_state_dict(params, strict=True)
    m = m.eval().to(DEV).to(dtype)
    if mode in ("fma", "x6"):
        m.__dict__["_nmm_fp32_fma" if mode == "fma" else "_nmm_fp32_exact"] = True
    with torch.no_grad():
        y = m(x.to(DEV, dtype), encoder_hidden_states=ctx.to(DEV, dtype)).sample
    ref = so.forward_reference_order({k: v.double() for k, v in params.items()}, x.double(), ctx.double(), cfg)
    err = (y.double().cpu() - ref).abs().max().item()
    if mode == "bf16":
        bound = TOL_BF16 + 2 ** -8 * ref.abs().max().item()
    else:
        bound = TOL_FP32 + 4 * ulp32(ref.abs().max().item())
    print(f"spatial {mode}: err {err:.2e} bound {bound:.2e}")
    assert math.isfinite(err) and err <= bound, (err, bound)


@pytest.mark.gpu
@pytest.mark.parametrize("C,side,dtype,ratio", [(320, 16, torch.bfloat16, 30), (640, 8, torch.bfloat16, 30), (320, 8, torch.float32, 300)])
def test_carried_y_sums_offset(C, side, dtype, ratio):
    """forward_packed(..., y_sums=...) on an offset x (y = x + ... keeps the offset): the variance the sums imply, against fp64 of y as
    stored.  The raw sum of squares is dominated by mean^2 and says nothing.  Relative bound: 1e-5 in fp32 (gn_stats over y), 2^-9 in bf16
    (rstd to half a bf16 ulp; C = 640 takes its sums from proj_out's epilogue)."""
    from neurons_b200 import ops
    from tests import helpers
    B, F = 1, 8
    cfg, params, x, _ = _module_case(C, F, side, B, ratio, seed=C + 1, dtype=dtype)
    m = helpers.mirror_module(cfg, params, DEV, dtype)
    xd = x.to(DEV, dtype)
    with torch.no_grad():
        m(xd, None, None)
        eng = m.__dict__["_nmm_engine"]
        y_sums = torch.full((B * F * 32, 2), float("nan"), dtype=torch.float64, device=DEV)
        y = ops.forward_packed(xd, eng.packed, eng.cfg, y_sums=y_sums)
    n = (C // GROUPS) * side * side
    s = y_sums.cpu()
    var = s[:, 1] / n - (s[:, 0] / n) ** 2
    _, v64, _ = group_stats64(y.cpu())
    rel = ((var - v64.reshape(-1)) / v64.reshape(-1)).abs().max().item()
    assert rel <= (1e-5 if dtype == torch.float32 else 2 ** -9), rel
