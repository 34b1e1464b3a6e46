"""The attention kernels at the edges of their online softmax, against fp64 on exactly the values each kernel receives.

Inputs with randn q and k give scaled logits of about N(0, 1): a flat softmax whose running max never moves far after the first key tile.
The constructors here aim at what a flash-style kernel can get wrong instead.  For every (image, head) a unit direction u is drawn; queries
are sigma_i * alpha * u (+ small noise) with the row pattern sigma_i = +1, 0, -1 (period 3, so that neighbouring rows, both query tiles of a
two-tile CTA and both halves of a row split over two threads behave differently), keys are small noise plus beta_j * u on chosen keys, so
that the logit of key j in a sigma = +1 row is beta_j (in log2 units below: level b_j, beta_j = b_j ln 2):

  jump        one key `at` lies J log2 units above all the others: the tcgen05 kernel keeps a per-row REFERENCE max and rescales O in tensor
              memory only when a later tile's max is more than 2^8 above it (spatial_attention_tc.cu), J straddles that threshold
  staircase   every 128-key tile's max 9 log2 units above the previous one: the rescale on every tile
  descending  tile 0 holds the max, later tiles >= 130 log2 units lower: underflow, the -125 clamp of the polynomial exp2; sigma = -1 rows
              see the mirror image (one raise of >= 130 at tile 1, O's row scaled to zero)
  offset      +-c natural logit units added to whole rows (a channel of q against a constant channel of k): softmax must not change
  uniform     q = 0: O is the mean of the valid V rows (V with a non-zero mean), the masked keys of a ragged last tile must not dilute it
  peaked      randn q scaled to a given max |logit|

The CPU tests check that the constructors do what they claim (an fp64 replay of the tcgen05 raise rule) and that the bf16 bound used on
the GPU would catch a broken rescale (a float emulation of the lazy-max softmax passes it, its mutants fail it by >= 10x).  The GPU tests
run every hand-written attention path on them: the tcgen05 spatial kernels (default two-tile and the A/B variants), the mma.sync kernels,
the fp32 checker, the fp32-grade x3 kernel (also against an fp64 emulation of its own arithmetic), the temporal attention variants, the
QKV projection with attention in its epilogue and the video decoder's temporal attention.
"""
import math

import pytest
import torch

from tests.helpers import round_bf16

LOG2E = 1.4426950408889634
TILE = 128                  # keys per tile of the tcgen05 kernels
SIGMA = (1.0, 0.0, -1.0)
EPS = 0.01                  # noise on q and k of the direction-built cases


# ---- constructors ------------------------------------------------------------------------------------------------------------------
def _sigma(Lq):
    return torch.tensor([SIGMA[i % 3] for i in range(Lq)], dtype=torch.float64)


def _levels(kind, Lkv, J=None, at=None):
    """Key levels b_j in log2 units (logit of key j in a sigma = +1 row = b_j ln 2)."""
    j = torch.arange(Lkv)
    if kind == "jump":
        b = torch.zeros(Lkv, dtype=torch.float64)
        b[at] = J
        return b
    if kind == "staircase":
        return 9.0 * (j // TILE).double()
    if kind == "descending":
        return torch.where(j < TILE, 0.0, -130.0 - (j // TILE).double())
    raise ValueError(kind)


def make_case(kind, Lq, Lkv, heads, dh, images=2, kv_div=1, seed=0, J=None, at=None, c=None, logit=None):
    """-> fp32 q [images, Lq, heads * dh], k, v [images / kv_div, Lkv, heads * dh] (not rounded: callers round to what the kernel takes)."""
    g = torch.Generator().manual_seed(seed)
    C, KI = heads * dh, images // kv_div
    v = torch.randn(KI, Lkv, heads, dh, generator=g, dtype=torch.float64)
    if kind in ("jump", "staircase", "descending"):
        u = torch.randn(KI, heads, dh, generator=g, dtype=torch.float64)
        u = u / u.norm(dim=-1, keepdim=True)
        beta = _levels(kind, Lkv, J, at) * math.log(2.0)
        k = beta.view(1, Lkv, 1, 1) * u.unsqueeze(1) + EPS * torch.randn(KI, Lkv, heads, dh, generator=g, dtype=torch.float64)
        uq = u.repeat_interleave(kv_div, dim=0)
        q = (_sigma(Lq).view(1, Lq, 1, 1) * math.sqrt(dh)) * uq.unsqueeze(1) + EPS * torch.randn(images, Lq, heads, dh, generator=g, dtype=torch.float64)
        v = v + (1.0 - 2.0 * ((torch.arange(Lkv) // TILE) % 2).double()).view(1, Lkv, 1, 1)        # tile means +1, -1, ...: weights off by
    elif kind == "offset":
        q = 0.5 * torch.randn(images, Lq, heads, dh, generator=g, dtype=torch.float64)
        k = torch.randn(KI, Lkv, heads, dh, generator=g, dtype=torch.float64)
        k[..., 0] = 1.0
        q[..., 0] = _sigma(Lq).view(1, Lq, 1) * c * math.sqrt(dh)
    elif kind == "uniform":
        q = torch.zeros(images, Lq, heads, dh, dtype=torch.float64)
        k = torch.randn(KI, Lkv, heads, dh, generator=g, dtype=torch.float64)
        v = 1.5 + 0.5 * v
    elif kind == "peaked":
        q = torch.randn(images, Lq, heads, dh, generator=g, dtype=torch.float64)
        k = torch.randn(KI, Lkv, heads, dh, generator=g, dtype=torch.float64)
        s = torch.einsum("iqhd,ikhd->ihqk", q, k.repeat_interleave(kv_div, dim=0)) / math.sqrt(dh)
        q = q * (logit / s.abs().max().item())
    else:
        raise ValueError(kind)
    return q.reshape(images, Lq, C).float(), k.reshape(KI, Lkv, C).float(), v.reshape(KI, Lkv, C).float()


def _heads(t, heads):
    """[I, L, C] -> [I, heads, L, dh] float64."""
    I, L, C = t.shape
    return t.double().view(I, L, heads, C // heads).permute(0, 2, 1, 3)


def _merge(o):
    I, H, L, dh = o.shape
    return o.permute(0, 2, 1, 3).reshape(I, L, H * dh)


def attention_fp64(q, k, v, heads, kv_div=1):
    """softmax(q k^T / sqrt(d_h)) v per (image, head) in float64; q [I, Lq, C], k / v [I / kv_div, Lkv, C]."""
    qq = _heads(q, heads)
    kk, vv = (_heads(t, heads).repeat_interleave(kv_div, dim=0) for t in (k, v))
    p = torch.softmax(qq @ kk.transpose(-1, -2) * qq.shape[-1] ** -0.5, dim=-1)
    return _merge(p @ vv)


def _f32(x):
    return x.float().double()


def _scale_log2e(dh):
    """The kernels' fp32 constant: (1 / sqrtf(d_h)) * 1.4426950408889634f, both steps rounded to fp32."""
    s = torch.tensor(1.0 / math.sqrt(dh), dtype=torch.float32)
    return (s * torch.tensor(LOG2E, dtype=torch.float32)).double().item()


def _scores_f32(q, k, heads, kv_div=1):
    qq = _heads(q, heads)
    kk = _heads(k, heads).repeat_interleave(kv_div, dim=0)
    return _f32(qq @ kk.transpose(-1, -2))


def replay_raises(q, k, heads, kv_div=1):
    """fp64 replay of the tcgen05 kernels' reference-max rule on the values they receive: per 128-key tile, raise the row's reference max
    when (tile max - reference) * scale * log2 e > 8.  -> bool [I, heads, Lq, tiles] (tile 0 always raises)."""
    s = _scores_f32(q, k, heads, kv_div)
    sl = _scale_log2e(q.shape[-1] // heads)
    Lkv = s.shape[-1]
    m_ref = torch.full(s.shape[:-1], -math.inf, dtype=torch.float64)
    out = []
    for t in range((Lkv + TILE - 1) // TILE):
        mx = s[..., t * TILE:(t + 1) * TILE].max(-1).values
        r = (mx - m_ref) * sl > 8.0
        m_ref = torch.where(r, mx, m_ref)
        out.append(r)
    return torch.stack(out, -1)


def lazy_softmax_attention(q, k, v, heads, kv_div=1, mutant=None):
    """Float emulation of the tcgen05 kernels' softmax: fp32 scores, per 128-key tile the reference-max rule (threshold 2^8), bf16 weights
    p = 2^((s - m_ref) * scale * log2 e), O and the row sum (the ones column of V) accumulated in fp64, O's row and its sum rescaled on a
    raise.  mutant: "skip" = no rescale at all, "no_sum" = O rescaled but not the row sum."""
    s = _scores_f32(q, k, heads, kv_div)
    vv = _heads(v, heads).repeat_interleave(kv_div, dim=0)
    sl = _scale_log2e(q.shape[-1] // heads)
    Lkv = s.shape[-1]
    m_ref = torch.full(s.shape[:-1], -math.inf, dtype=torch.float64)
    O = torch.zeros(s.shape[:-1] + (vv.shape[-1],), dtype=torch.float64)
    l = torch.zeros(s.shape[:-1], dtype=torch.float64)
    for t in range((Lkv + TILE - 1) // TILE):
        st = s[..., t * TILE:(t + 1) * TILE]
        mx = st.max(-1).values
        r = (mx - m_ref) * sl > 8.0
        m_new = torch.where(r, mx, m_ref)
        if t > 0 and mutant != "skip":
            f = torch.exp2((m_ref - m_new) * sl)
            O = O * f.unsqueeze(-1)
            if mutant != "no_sum":
                l = l * f
        p = torch.exp2((st - m_new.unsqueeze(-1)) * sl).to(torch.bfloat16).double()
        O = O + p @ vv[..., t * TILE:(t + 1) * TILE, :]
        l = l + p.sum(-1)
        m_ref = m_new
    return _merge(O / l.unsqueeze(-1))


def _split(x):
    """fp32 -> (hi, lo) bf16 planes as float64: the NMM_F32X3 operand split."""
    x = x.float()
    hi = x.to(torch.bfloat16)
    return hi.double(), (x - hi.float()).to(torch.bfloat16).double()


def x3_emulation(q, k, v, heads, kv_div=1):
    """fp64 emulation of the fp32-grade spatial attention (spatial_attention_x3.cu): q, k, v split into bf16 hi + lo, S = Qh Kh + Qh Kl +
    Ql Kh rounded to fp32, an online softmax over 64-key tiles with fp32 exponent arguments, the weights split into hi + lo and O += Ph Vh +
    Ph Vl + Pl Vh, the row sum over the fp32 weights.  What it leaves out is the order of the fp32 accumulations inside the MMAs."""
    qh, ql = (_heads(t, heads) for t in _split(q))
    kh, kl = (_heads(t, heads).repeat_interleave(kv_div, dim=0) for t in _split(k))
    vh, vl = (_heads(t, heads).repeat_interleave(kv_div, dim=0) for t in _split(v))
    S = _f32(qh @ kh.transpose(-1, -2) + qh @ kl.transpose(-1, -2) + ql @ kh.transpose(-1, -2))
    sl = _scale_log2e(q.shape[-1] // heads)
    Lkv = S.shape[-1]
    m = torch.full(S.shape[:-1], -math.inf, dtype=torch.float64)
    O = torch.zeros(S.shape[:-1] + (vh.shape[-1],), dtype=torch.float64)
    l = torch.zeros(S.shape[:-1], dtype=torch.float64)
    for t in range((Lkv + 63) // 64):
        sel = slice(t * 64, (t + 1) * 64)
        st = S[..., sel]
        mx = torch.maximum(m, st.max(-1).values)
        al = _f32(torch.exp2(_f32((m - mx) * sl)))
        e = _f32(torch.exp2(_f32(st * sl - _f32(mx * sl).unsqueeze(-1))))
        ph, pl = _split(e)
        l = l * al + e.sum(-1)
        O = O * al.unsqueeze(-1) + ph @ vh[..., sel, :] + ph @ vl[..., sel, :] + pl @ vh[..., sel, :]
        m = mx
    return _merge(O / l.unsqueeze(-1))


def _score_rounding(q, k, heads, kv_div=1):
    """Scale of the fp32 rounding in the scores, in natural logit units: 4 ulps-worth of the largest absolute-value sum sum_d |q_d k_d| / sqrt(d_h)
    (the terms' magnitude, not the logit's, sets the accumulation error: an offset row of 200 has scores exact to ~2^-24 * 200 only)."""
    qq = _heads(q, heads).abs()
    kk = _heads(k, heads).abs().repeat_interleave(kv_div, dim=0)
    return 2.0 ** -22 * (qq @ kk.transpose(-1, -2)).max().item() * qq.shape[-1] ** -0.5


def _maxabs(a, b):
    return (a.double().cpu() - b.double().cpu()).abs().max().item()


def tol_bf16(v):
    """bf16 kernels: exact inputs, fp32 scores, P and O rounded to bf16 -> half an ulp of O plus the weights' rounding (the row sum adds the
    rounded weights, so O / l is an exact weighted mean): 2^-8 of max |v| (the bound of test_gpu_parity.py)."""
    return 2.0 ** -8 * 1.01 * v.abs().max().item()


def tol_fp32(q, k, v, heads, kv_div=1):
    """fp32 kernels: 2e-5 of max(1, max |v|), plus what the fp32 rounding of the scores does to a weighted mean (twice its logit error)."""
    mv = v.abs().max().item()
    return 2e-5 * max(1.0, mv) + 2.0 * mv * _score_rounding(q, k, heads, kv_div)


# ---- the case lists ----------------------------------------------------------------------------------------------------------------
JUMPS = (7.9, 8.0, 8.1, 8.5, 12.0, 40.0, 200.0)


def jump_positions(Lkv):
    """first key of tile 1; key 64 of a middle tile (the second half of a row split over two threads); key 127 of a tile; the last key
    (of a ragged last tile when Lkv % 128 != 0)."""
    nt = (Lkv + TILE - 1) // TILE
    return {"t1": TILE, "k64": TILE * max(1, nt // 2) + 64, "k127": TILE * max(1, nt - 2) + 127, "last": Lkv - 1}


def case_kw(case, Lkv):
    """'jump40@t1' / 'offset100' / 'peaked30' / 'staircase' ... -> make_case kwargs."""
    if case.startswith("jump"):
        J, name = case[4:].split("@")
        return dict(kind="jump", J=float(J), at=jump_positions(Lkv)[name])
    for kind, arg in (("offset", "c"), ("peaked", "logit")):
        if case.startswith(kind):
            return {"kind": kind, arg: float(case[len(kind):])}
    return dict(kind=case)


def cases(Lkv, jumps=JUMPS, ats=None, offsets=(30.0, 100.0, 200.0), peaks=(10.0, 30.0, 60.0)):
    """-> [(id, make_case kwargs)] for one key length."""
    out = []
    pos = jump_positions(Lkv)
    for name in (pos if ats is None else ats):
        for J in jumps:
            out.append((f"jump{J:g}@{name}", dict(kind="jump", J=J, at=pos[name])))
    out += [("staircase", dict(kind="staircase")), ("descending", dict(kind="descending")), ("uniform", dict(kind="uniform"))]
    out += [(f"offset{c:g}", dict(kind="offset", c=c)) for c in offsets]
    out += [(f"peaked{p:g}", dict(kind="peaked", logit=p)) for p in peaks]
    return out


# ---- CPU: the constructors do what they claim; the bound catches a broken rescale ----------------------------------------------------
def _bf16_case(**kw):
    q, k, v = make_case(**kw)
    return round_bf16(q), round_bf16(k), round_bf16(v)


@pytest.mark.parametrize("dh", [40, 80])
@pytest.mark.parametrize("Lkv", [300, 1024])
@pytest.mark.parametrize("J", JUMPS)
def test_jump_raises_where_intended(dh, Lkv, J):
    Lq, heads = 96, 2
    for name, at in jump_positions(Lkv).items():
        q, k, v = _bf16_case(kind="jump", Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, J=J, at=at, seed=Lkv + dh)
        r = replay_raises(q, k, heads)
        sig = _sigma(Lq)
        later = r[..., 1:]
        assert not later[..., sig != 1, :].any(), (name, "sigma 0 / -1 rows must never raise after tile 0")
        plus = later[..., sig == 1, :]
        if J <= 7.9:
            assert not plus.any(), name
        elif J >= 8.1:
            want = torch.zeros(later.shape[-1], dtype=torch.bool)
            want[at // TILE - 1] = True
            assert (plus == want).all(), (name, J)
        # the keys before the jump's tile carry the mass the rescale must carry (a skipped / wrong rescale is then an O(1) error), and
        # the keys other than the jump key most of it where there are more of them than 2^J
        p = torch.softmax(_scores_f32(q, k, heads).mul(dh ** -0.5)[..., sig == 1, :], -1)
        if J <= 8.5:
            assert p[..., :at // TILE * TILE].sum(-1).min().item() >= 0.05, name
            if Lkv - 1 >= 2 * 2 ** J:
                assert (1.0 - p[..., at]).min().item() >= 0.5, name


@pytest.mark.parametrize("dh", [40, 80])
@pytest.mark.parametrize("Lkv", [256, 383, 1024])
def test_staircase_and_descending_raise_where_intended(dh, Lkv):
    Lq, heads = 96, 2
    sig = _sigma(Lq)
    q, k, _ = _bf16_case(kind="staircase", Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, seed=3)
    r = replay_raises(q, k, heads)
    assert r[..., sig == 1, :].all()                                  # every tile raises
    assert not r[..., sig != 1, 1:].any()
    q, k, _ = _bf16_case(kind="descending", Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, seed=4)
    r = replay_raises(q, k, heads)
    assert not r[..., sig == 1, 1:].any()
    assert r[..., sig == -1, 1].all() and not r[..., sig == -1, 2:].any()
    s = _scores_f32(q, k, heads) * _scale_log2e(dh)
    gap = s[..., sig == 1, :TILE].max(-1).values - s[..., sig == 1, TILE:].max(-1).values
    assert gap.min().item() >= 130.0                                  # later tiles underflow (and hit the -125 clamp of the polynomial exp2)


def test_offset_and_uniform_constructors():
    heads, dh = 2, 40
    q, k, v = _bf16_case(kind="offset", Lq=30, Lkv=300, heads=heads, dh=dh, c=100.0)
    q0, k0, _ = _bf16_case(kind="offset", Lq=30, Lkv=300, heads=heads, dh=dh, c=0.0)
    s, s0 = (_heads(a, heads) @ _heads(b, heads).transpose(-1, -2) * dh ** -0.5 for a, b in ((q, k), (q0, k0)))
    d = s - s0                                                        # a constant per row: +-100 (sigma = +-1), 0
    assert (d.max(-1).values - d.min(-1).values).abs().max().item() < 1e-9
    assert abs(d[..., 0, :].mean().item() - 100.0) < 0.5 and abs(d[..., 2, :].mean().item() + 100.0) < 0.5
    assert torch.allclose(attention_fp64(q, k, v, heads), attention_fp64(q0, k0, v, heads), atol=1e-12)
    q, k, v = _bf16_case(kind="uniform", Lq=30, Lkv=257, heads=heads, dh=dh)
    assert torch.allclose(attention_fp64(q, k, v, heads), v.double().mean(1, keepdim=True).expand(2, 30, -1), atol=1e-12)
    assert v.mean().item() > 1.0                                      # diluting with masked (zero) V rows would be visible


@pytest.mark.parametrize("case", ["jump8.5", "jump12", "jump40", "staircase", "descending", "uniform"])
@pytest.mark.parametrize("dh", [40, 80])
def test_lazy_softmax_emulation_passes_and_its_mutants_fail(case, dh):
    Lq, Lkv, heads = 96, 1024 if case != "uniform" else 383, 2
    kw = dict(kind="jump", J=float(case[4:]), at=TILE) if case.startswith("jump") else dict(kind=case)
    q, k, v = _bf16_case(Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, seed=11, **kw)
    ref = attention_fp64(q, k, v, heads)
    tol = tol_bf16(v)
    good = _maxabs(lazy_softmax_attention(q, k, v, heads), ref)
    assert good <= tol / 3, (good, tol)
    if case in ("descending", "uniform"):
        return                                                        # no raise after tile 0 in the sigma = +1 rows: nothing to mutate
    for mutant in ("skip", "no_sum"):
        bad = _maxabs(lazy_softmax_attention(q, k, v, heads, mutant=mutant), ref)
        assert bad >= 10 * tol, (mutant, bad, tol)


def test_x3_emulation_tracks_fp64_at_flat_logits():
    """At N(0, 1) logits the emulated x3 arithmetic is within the module-level fp32 figure (2.5e-5) of fp64."""
    q, k, v = make_case("peaked", 64, 300, 2, 40, logit=4.0)
    assert _maxabs(x3_emulation(q, k, v, 2), attention_fp64(q, k, v, 2)) <= 1e-5


# ---- GPU ---------------------------------------------------------------------------------------------------------------------------
def _gpu():
    import neurons_b200 as nb
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return nb


def _spatial(q, k, v, heads, kv_div, dtype, variant=0, x3=False):
    nb = _gpu()
    from neurons_b200 import lib as nlib
    with nlib.options({nlib.OPT_SPATIAL_ATTN: variant}):
        o = nb.spatial_attention(q.cuda().to(dtype), k.cuda().to(dtype), v.cuda().to(dtype), heads, kv_div, x3=x3)
        torch.cuda.synchronize()
    return o.cpu()


def _check_bf16(kw, Lq, Lkv, dh, variant=0, images=2, heads=2, kv_div=1):
    q, k, v = _bf16_case(Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, images=images, kv_div=kv_div, seed=Lq + Lkv + dh, **kw)
    o = _spatial(q, k, v, heads, kv_div, torch.bfloat16, variant)
    err = _maxabs(o, attention_fp64(q, k, v, heads, kv_div))
    tol = tol_bf16(v)
    assert math.isfinite(err) and err <= tol, (err, tol)


# the default tcgen05 kernel (two 128-query tiles per CTA): every case at every key length, ragged query counts
TC_SHAPES = [(256, 256), (257, 257), (300, 300), (383, 383), (200, 384), (513, 513), (300, 1024), (130, 4096)]       # (Lq, Lkv)


def _tc_params():
    out = []
    for Lq, Lkv in TC_SHAPES:
        full = Lkv in (300, 1024)
        for cid, kw in cases(Lkv, jumps=JUMPS if full else (8.5, 200.0), ats=None if full else ("t1", "last"),
                             offsets=(30.0, 100.0, 200.0) if full else (200.0,), peaks=(10.0, 30.0, 60.0) if full else (30.0,)):
            for dh in (40, 80):
                out.append(pytest.param(kw, Lq, Lkv, dh, id=f"{cid}-Lq{Lq}-Lkv{Lkv}-dh{dh}"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kw,Lq,Lkv,dh", _tc_params())
def test_tcgen05_two_tile_default(kw, Lq, Lkv, dh):
    _check_bf16(kw, Lq, Lkv, dh)


# A/B variants of the tcgen05 kernel with correct results (15, 17, 26 drop K / V traffic on purpose; >= 100 is the trace build's)
TC_VARIANTS = [2, 3, 10, 11, 12, 13, 14, 16, 20, 22, 27]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", TC_VARIANTS)
@pytest.mark.parametrize("case", ["jump8.5@k64", "jump40@t1", "jump200@last", "staircase", "uniform"])
@pytest.mark.parametrize("Lq,Lkv,dh", [(300, 300, 40), (257, 1024, 80), (383, 383, 80)])
def test_tcgen05_variants(variant, case, Lq, Lkv, dh):
    _check_bf16(case_kw(case, Lkv), Lq, Lkv, dh, variant=variant)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["jump40@last", "uniform", "peaked30", "offset100"])
@pytest.mark.parametrize("dh", [40, 80])
def test_tcgen05_text_cross_attention(case, dh):
    """NMM_OPT_SPATIAL_ATTN = 24: the 77-token text cross-attention (kv image = image / frames) on the two-tile kernel."""
    _check_bf16(case_kw(case, 77), 300, 77, dh, variant=24, images=4, kv_div=2)


# mma.sync kernels: variant 1 forces them at d_h 40 / 80; <= 128 keys -> the 4-warp kernel unless variant 25; d_h 160 always
MMA_SHAPES = [(300, 300, 40, 1, 1), (257, 1024, 80, 1, 1), (200, 384, 160, 1, 1), (300, 77, 40, 1, 2), (300, 77, 160, 0, 2),
              (300, 77, 80, 25, 2), (100, 128, 80, 1, 1), (100, 129, 160, 0, 1)]      # (Lq, Lkv, dh, variant, kv_div)


def _mma_params():
    out = []
    for Lq, Lkv, dh, variant, kv_div in MMA_SHAPES:
        for cid, kw in cases(Lkv, jumps=(8.5, 40.0, 200.0), ats=("t1", "last") if Lkv > TILE else (), offsets=(200.0,), peaks=(30.0, 60.0)):
            out.append(pytest.param(kw, Lq, Lkv, dh, variant, kv_div, id=f"{cid}-Lq{Lq}-Lkv{Lkv}-dh{dh}-v{variant}-kvdiv{kv_div}"))
        if Lkv <= TILE:
            out.append(pytest.param(dict(kind="jump", J=40.0, at=Lkv - 1), Lq, Lkv, dh, variant, kv_div, id=f"jump40@last-Lq{Lq}-Lkv{Lkv}-dh{dh}-v{variant}"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kw,Lq,Lkv,dh,variant,kv_div", _mma_params())
def test_mma_sync_kernels(kw, Lq, Lkv, dh, variant, kv_div):
    _check_bf16(kw, Lq, Lkv, dh, variant=variant, images=2 * kv_div, kv_div=kv_div)


# fp32 checker (one warp per query, fp32 throughout): small shapes
F32_SHAPES = [(100, 300, 40, 1), (64, 257, 80, 1), (50, 130, 160, 1), (60, 77, 40, 2)]


def _f32_params():
    out = []
    for Lq, Lkv, dh, kv_div in F32_SHAPES:
        for cid, kw in cases(Lkv, jumps=(8.5, 40.0, 200.0), ats=("t1", "last") if Lkv > TILE else ()):
            out.append(pytest.param(kw, Lq, Lkv, dh, kv_div, id=f"{cid}-Lq{Lq}-Lkv{Lkv}-dh{dh}-kvdiv{kv_div}"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kw,Lq,Lkv,dh,kv_div", _f32_params())
def test_fp32_checker_kernel(kw, Lq, Lkv, dh, kv_div):
    heads = 2
    q, k, v = make_case(Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, images=2 * kv_div, kv_div=kv_div, seed=Lkv + dh, **kw)
    o = _spatial(q, k, v, heads, kv_div, torch.float32)
    err = _maxabs(o, attention_fp64(q, k, v, heads, kv_div))
    tol = tol_fp32(q, k, v, heads, kv_div)
    assert err <= tol, (err, tol)


# fp32-grade x3 kernel through its own entry
X3_SHAPES = [(100, 300, 40, 1), (130, 1024, 80, 1), (64, 257, 160, 1), (100, 77, 40, 2), (64, 77, 160, 2)]


def _x3_params():
    out = []
    for Lq, Lkv, dh, kv_div in X3_SHAPES:
        for cid, kw in cases(Lkv, jumps=(8.5, 40.0, 200.0), ats=("t1", "last") if Lkv > TILE else ()):
            out.append(pytest.param(kw, Lq, Lkv, dh, kv_div, id=f"{cid}-Lq{Lq}-Lkv{Lkv}-dh{dh}-kvdiv{kv_div}"))
    return out


def x3_tol_vs_emulation(q, k, v, heads, kv_div=1):
    """What the emulation leaves out: the order of the fp32 accumulations of O and l (1e-5) and of S (2 ulps of the terms' magnitude in
    logits, twice over |v|; the emulation rounds S once)."""
    return 1e-5 + v.abs().max().item() * _score_rounding(q, k, heads, kv_div)


@pytest.mark.gpu
@pytest.mark.parametrize("kw,Lq,Lkv,dh,kv_div", _x3_params())
def test_x3_kernel(kw, Lq, Lkv, dh, kv_div):
    heads = 2
    q, k, v = make_case(Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, images=2 * kv_div, kv_div=kv_div, seed=Lkv + dh, **kw)
    o = _spatial(q, k, v, heads, kv_div, torch.float32, x3=True)
    assert o.dtype == torch.float32
    emu = x3_emulation(q, k, v, heads, kv_div)
    ref = attention_fp64(q, k, v, heads, kv_div)
    tol = x3_tol_vs_emulation(q, k, v, heads, kv_div)
    err_emu = _maxabs(o, emu)
    assert err_emu <= tol, ("kernel vs emulation of its arithmetic", err_emu, tol)
    # against fp64: the error the design predicts (the emulation's own error grows with the logits: no fixed 1e-4 here)
    predicted = _maxabs(emu, ref)
    err = _maxabs(o, ref)
    assert err <= predicted + tol, ("kernel vs fp64", err, predicted, tol)


@pytest.mark.gpu
@pytest.mark.parametrize("dh,kv_div,Lq,Lkv", [(40, 1, 300, 300), (80, 1, 256, 256), (160, 1, 200, 200), (40, 2, 300, 77), (80, 4, 100, 77)])
def test_x3_kernel_flat_logits_vs_fp64(dh, kv_div, Lq, Lkv):
    """randn q, k, v (N(0, 1) logits): x3=True agrees with fp64 to within the module-level fp32-mode figure, 2.5e-5."""
    heads = 8 if dh < 160 else 4
    g = torch.Generator().manual_seed(dh + Lkv)
    q = torch.randn(2 * kv_div, Lq, heads * dh, generator=g)
    k, v = torch.randn(2, 2, Lkv, heads * dh, generator=g)
    o = _spatial(q, k, v, heads, kv_div, torch.float32, x3=True)
    err = _maxabs(o, attention_fp64(q, k, v, heads, kv_div))
    assert err <= 2.5e-5, err


@pytest.mark.gpu
def test_options_select_the_intended_kernels():
    """The option values above reach the kernels they are meant to test (kernel names from torch.profiler)."""
    nb = _gpu()
    from neurons_b200 import lib as nlib
    from torch.profiler import ProfilerActivity, profile

    def names(variant, Lq, Lkv, dh, kv_div=1, dtype=torch.bfloat16, x3=False):
        q, k, v = make_case("uniform", Lq, Lkv, 2, dh, images=2 * kv_div, kv_div=kv_div)
        q, k, v = (t.cuda().to(dtype) for t in (q, k, v))
        with nlib.options({nlib.OPT_SPATIAL_ATTN: variant}):
            nb.spatial_attention(q, k, v, 2, kv_div, x3=x3)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                nb.spatial_attention(q, k, v, 2, kv_div, x3=x3)
                torch.cuda.synchronize()
        return " ".join(e.key for e in prof.key_averages() if "attention" in e.key)

    assert "spatial_attention_tc2_kernel<40, 3, false, false>" in names(0, 300, 300, 40)
    assert "spatial_attention_tc2_kernel<80, 2, false, false>" in names(0, 300, 300, 80)
    assert "spatial_attention_tc2_kernel<40, 3, false, true>" in names(27, 300, 300, 40)
    assert "spatial_attention_tc2_kernel<80, 2, false, false>" in names(24, 300, 77, 80, kv_div=2)
    assert "spatial_attention_tc_kernel<40, 2, 3" in names(2, 300, 300, 40)
    assert "spatial_attention_tc_kernel<80, 1, 6" in names(14, 300, 300, 80)
    assert "spatial_attention_tc_kernel<40, 1, 3, false, true>" in names(16, 300, 300, 40)
    assert "spatial_attention_kernel<40, 8>" in names(1, 300, 300, 40)
    assert "spatial_attention_kernel<80, 4>" in names(1, 300, 77, 80, kv_div=2)
    assert "spatial_attention_kernel<80, 8>" in names(25, 300, 77, 80, kv_div=2)
    assert "spatial_attention_kernel<160, 8>" in names(0, 200, 384, 160)
    assert "spatial_attention_f32_kernel<40>" in names(0, 100, 300, 40, dtype=torch.float32)
    assert "spatial_attention_x3_kernel<80>" in names(0, 100, 300, 80, dtype=torch.float32, x3=True)


# ---- temporal attention (attention over the frames of a position) ----------------------------------------------------------------
def _temporal_case(kind, F, C, heads, P, B=1, seed=0):
    """qkv [B * F * P, 3C] in the (b, f, p) token order of the motion module; the attention runs over f per (b, p, head)."""
    g = torch.Generator().manual_seed(seed)
    dh = C // heads
    z = torch.randn(B, F, P, 3, heads, dh, generator=g, dtype=torch.float64)
    sig = _sigma(P).view(1, 1, P, 1)
    if kind.startswith("offset"):
        c = float(kind[6:])
        z[:, :, :, 0] *= 0.5
        z[:, :, :, 1, :, 0] = 1.0
        z[:, :, :, 0, :, 0] = sig * c * math.sqrt(dh)
    elif kind.startswith("peaked"):
        s = torch.einsum("bfphd,bgphd->bphfg", z[:, :, :, 0], z[:, :, :, 1]) * dh ** -0.5
        z[:, :, :, 0] *= float(kind[6:]) / s.abs().max().item()
    elif kind == "uniform":
        z[:, :, :, 0] = 0.0
        z[:, :, :, 2] = 1.5 + 0.5 * z[:, :, :, 2]
    elif kind.startswith("dominant"):                                 # frame F // 3 of every key set J log2 units above the others
        J = float(kind[8:])
        u = torch.randn(B, 1, P, heads, dh, generator=g, dtype=torch.float64)
        u = u / u.norm(dim=-1, keepdim=True)
        lev = torch.zeros(F, dtype=torch.float64)
        lev[F // 3] = J * math.log(2.0)
        z[:, :, :, 1] = lev.view(1, F, 1, 1, 1) * u + EPS * z[:, :, :, 1]
        z[:, :, :, 0] = sig.unsqueeze(-1) * math.sqrt(dh) * u + EPS * z[:, :, :, 0]
    else:
        raise ValueError(kind)
    return z.reshape(B * F * P, 3 * C).float()


def _temporal_fp64(qkv, B, F, P, heads):
    C = qkv.shape[1] // 3
    dh = C // heads
    z = qkv.double().reshape(B, F, P, 3, heads, dh)
    s = torch.einsum("bfphd,bgphd->bphfg", z[:, :, :, 0], z[:, :, :, 1]) * dh ** -0.5
    return torch.einsum("bphfg,bgphd->bfphd", s.softmax(-1), z[:, :, :, 2]).reshape(B * F * P, C)


TEMPORAL_KINDS = ["offset30", "offset100", "offset200", "peaked10", "peaked30", "peaked60", "uniform", "dominant12", "dominant200"]


@pytest.mark.gpu
@pytest.mark.parametrize("kind", TEMPORAL_KINDS)
@pytest.mark.parametrize("F,C", [(8, 320), (16, 640), (24, 1280), (32, 320)])
@pytest.mark.parametrize("variant", [0, 1, 2])
@pytest.mark.parametrize("dtype", [torch.bfloat16, torch.float32], ids=["bf16", "fp32"])
def test_temporal_attention_edges(kind, F, C, variant, dtype):
    nb = _gpu()
    from neurons_b200 import lib as nlib
    from neurons_b200 import ops
    from oracle import motion_oracle as mo
    heads, P, B = 8, 9, 1
    qkv = _temporal_case(kind, F, C, heads, P, B, seed=F + C)
    if dtype == torch.bfloat16:
        qkv = round_bf16(qkv)
    c = mo.MotionConfig(C, max_len=32)
    cfg = nb.ModuleConfig(c.channels, c.heads, c.layers, c.attn_blocks, c.pos_enc, c.max_len)
    with nlib.options({nlib.OPT_ATTN_VARIANT: variant}):
        ctx = ops.temporal_attention(cfg, (B, F, 3, 3), qkv.cuda().to(dtype))
        torch.cuda.synchronize()
    ref = _temporal_fp64(qkv, B, F, P, heads)
    v = qkv[:, 2 * C:]
    if dtype == torch.bfloat16:
        tol = tol_bf16(v)
    else:
        z = qkv.double().abs().reshape(B, F, P, 3, heads, C // heads)
        rnd = 2.0 ** -22 * torch.einsum("bfphd,bgphd->bphfg", z[:, :, :, 0], z[:, :, :, 1]).max().item() * (C // heads) ** -0.5
        tol = 2e-5 * max(1.0, v.abs().max().item()) + 2.0 * v.abs().max().item() * rnd
    err = _maxabs(ctx, ref)
    assert math.isfinite(err) and err <= tol, (err, tol)


def _exact_operands(N, C, seed):
    """Integer tokens in [-3, 3] and weights with 4 non-zeros per row from {+-1/4, +-1/2, +-1}: q, k, v = tokens . W^T are multiples of 1/4 of
    magnitude <= 12, exact in bf16, so the fused kernel, the two-kernel path and fp64 all see identical q, k, v."""
    g = torch.Generator().manual_seed(seed)
    tok = torch.randint(-3, 4, (N, C), generator=g).float()
    w = torch.zeros(3 * C, C)
    vals = torch.tensor([0.25, 0.5, 1.0])
    for r in range(3 * C):
        cols = torch.randperm(C, generator=g)[:4]
        w[r, cols] = vals[torch.randint(0, 3, (4,), generator=g)] * (torch.randint(0, 2, (4,), generator=g) * 2 - 1)
    return tok, w


@pytest.mark.gpu
@pytest.mark.parametrize("C,F,H,W,B", [(320, 8, 4, 4, 1), (320, 16, 4, 2, 2), (640, 16, 4, 4, 1), (640, 8, 8, 4, 1)])     # H*W % (128 / F) == 0
def test_qkv_attention_exact_operands_peaked(C, F, H, W, B):
    """QKV projection with the temporal attention in its epilogue at peaked logits (|logit| up to ~20 natural units)."""
    nb = _gpu()
    from neurons_b200 import lib as nlib
    from neurons_b200 import ops
    from oracle import motion_oracle as mo
    c = mo.MotionConfig(C, max_len=32)
    cfg = nb.ModuleConfig(c.channels, c.heads, c.layers, c.attn_blocks, c.pos_enc, c.max_len)
    P = H * W
    tok, w = _exact_operands(B * F * P, C, C + F)
    qkv = tok.double() @ w.double().T
    assert torch.equal(round_bf16(qkv.float()).double(), qkv)         # exact in bf16
    z = qkv.reshape(B, F, P, 3, c.heads, C // c.heads)
    logits = torch.einsum("bfphd,bgphd->bphfg", z[:, :, :, 0], z[:, :, :, 1]) * (C // c.heads) ** -0.5
    assert logits.abs().max().item() >= 10.0
    ref = _temporal_fp64(qkv, B, F, P, c.heads)
    tol = tol_bf16(qkv[:, 2 * C:])
    tokd, wd = tok.cuda().bfloat16(), w.cuda().bfloat16()
    fused = ops.qkv_attention(cfg, (B, F, H, W), tokd, wd)
    with nlib.options({nlib.OPT_ATTN_VARIANT: 0}):
        two = ops.temporal_attention(cfg, (B, F, H, W), ops.linear(tokd, wd, None, nlib.EPI_STORE))
    torch.cuda.synchronize()
    assert _maxabs(fused, ref) <= tol, (_maxabs(fused, ref), tol)
    assert _maxabs(two, ref) <= tol, (_maxabs(two, ref), tol)


@pytest.mark.gpu
@pytest.mark.parametrize("C,heads,side", [(64, 1, 5), (128, 4, 4), (128, 1, 7)])
def test_decoder_temporal_attention_peaked(C, heads, side):
    """The video decoder's temporal attention + blend (fp32) with to_q / to_k scaled for logits of about 30, against the oracle in fp64."""
    from neurons_b200 import video_decoder as vd
    from oracle import decoder_oracle as do
    from tests.test_video_decoder import FakeAttention
    from torch import nn
    import torch.nn.functional as TF
    cfg = do.DecoderAttnConfig(C, heads)
    params = do.make_params(cfg, C + heads)
    g = torch.Generator().manual_seed(side)
    x = torch.randn(6, C, side, side, generator=g)
    hs = x.reshape(1, 6, C, side * side).permute(0, 3, 1, 2).reshape(side * side, 6, C).double()
    hs = TF.group_norm(hs.transpose(1, 2), cfg.groups, params["group_norm.weight"].double(), params["group_norm.bias"].double(), cfg.eps).transpose(1, 2)
    dh = C // heads
    qq = TF.linear(hs, params["to_q.weight"].double(), params["to_q.bias"].double()).view(-1, 6, heads, dh)
    kk = TF.linear(hs, params["to_k.weight"].double(), params["to_k.bias"].double()).view(-1, 6, heads, dh)
    s = torch.einsum("nthd,nuhd->nhtu", qq, kk).abs().max().item() * dh ** -0.5
    f = (30.0 / s) ** 0.5
    for name in ("to_q.weight", "to_q.bias", "to_k.weight", "to_k.bias"):
        params[name] = params[name] * f
    attn = FakeAttention(cfg, params).cuda().eval()
    with torch.no_grad():
        y = vd.temporal_attention_blend(x.cuda(), attn, nn.Parameter(torch.tensor([0.3])).cuda(), 6)
        torch.cuda.synchronize()
        ref = do.temporal_blend_reference_order({k: t.double() for k, t in params.items()}, x.double(), 0.3, 6, cfg)
    err = _maxabs(y, ref)
    assert err <= 1e-4, err
