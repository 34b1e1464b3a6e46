"""The fp32 spatial attention of the FMA mode (NMM_F32) at every size: the tiled FMA-pipe flash kernel (spatial_attention_f32.cu) against
fp64 on the edge cases of test_attention_edges.py, side by side with the one-warp-per-query checker it replaces above the crossover, at the
UNet's full sizes through the default selection, and the spatial transformer in FMA mode at the config-2 64 x 64 level and at NEURONS'
16-frame 32 x 32 shape with self-attention logits of 30 to 60 (bar 1e-4 against the fp64 oracle)."""
import math

import pytest
import torch

from oracle import spatial_oracle as so
from tests.helpers import TOL_FP32
from tests.test_attention_edges import attention_fp64, case_kw, cases, make_case, tol_fp32

pytestmark = pytest.mark.gpu

TILED, CHECKER = 30, 31                 # NMM_OPT_SPATIAL_ATTN values that force the kernel of an fp32 call
F32_TILED_MIN_SCORES = 1 << 17          # launch_spatial_attention: Lq * Lkv * images * heads from which fp32 calls run the tiled kernel


def _run(q, k, v, heads, kv_div, variant):
    import neurons_b200 as nb
    from neurons_b200 import lib as nlib
    with nlib.options({nlib.OPT_SPATIAL_ATTN: variant}):
        o = nb.spatial_attention(q, k, v, heads, kv_div)
        torch.cuda.synchronize()
    return o


def _check(q, k, v, heads, kv_div, variant):
    o = _run(q.cuda(), k.cuda(), v.cuda(), heads, kv_div, variant).cpu()
    err = (o.double() - attention_fp64(q, k, v, heads, kv_div)).abs().max().item()
    tol = tol_fp32(q, k, v, heads, kv_div)
    assert math.isfinite(err) and err <= tol, (err, tol)
    return err


def _assert_default_runs(kernel, q, k, v, heads, kv_div=1):
    """The default selection runs `kernel` ("tiled" / "checker"): its output is bit-identical to the forced kernel's and differs from the
    other one's (both kernels are deterministic, their key orders differ), and torch.profiler names the kernel where it records kernels at
    all (in a long test process CUPTI may deliver none)."""
    from torch.profiler import ProfilerActivity, profile
    d = q.shape[-1] // heads
    want = f"spatial_attention_f32_tiled_kernel<{d}>" if kernel == "tiled" else f"spatial_attention_f32_kernel<{d}>"
    o = _run(q, k, v, heads, kv_div, 0)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _run(q, k, v, heads, kv_div, 0)
    names = " ".join(e.key for e in prof.key_averages() if "spatial_attention" in e.key)
    assert not names or want in names, (want, names)
    same, other = (TILED, CHECKER) if kernel == "tiled" else (CHECKER, TILED)
    assert torch.equal(o, _run(q, k, v, heads, kv_div, same))
    assert not torch.equal(o, _run(q, k, v, heads, kv_div, other))
    return o


# ---- the tiled kernel against fp64: every case kind, d_h 40 / 80 / 160, ragged tiles (64 / 128 / 32 queries, 32 keys), text cross-attention
TILED_SHAPES = [(100, 300, 40, 1), (257, 513, 80, 1), (130, 1024, 160, 1), (65, 33, 40, 1), (60, 77, 40, 2), (100, 77, 80, 8), (33, 77, 160, 2)]


def _tiled_params():
    out = []
    for Lq, Lkv, dh, kv_div in TILED_SHAPES:
        # every jump height and position at one shape, a subset at the others (<= 128 keys: no jump position past tile 0)
        kws = cases(Lkv) if (Lq, Lkv) == (100, 300) else cases(Lkv, jumps=(8.5, 40.0, 200.0), ats=("t1", "last") if Lkv > 128 else ())
        for cid, kw in kws:
            out.append(pytest.param(kw, Lq, Lkv, dh, kv_div, id=f"{cid}-Lq{Lq}-Lkv{Lkv}-dh{dh}-kvdiv{kv_div}"))
    return out


@pytest.mark.parametrize("kw,Lq,Lkv,dh,kv_div", _tiled_params())
def test_tiled_kernel_vs_fp64(kw, Lq, Lkv, dh, kv_div):
    heads = 2
    q, k, v = make_case(Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, images=2 * kv_div, kv_div=kv_div, seed=Lq + Lkv + dh, **kw)
    _check(q, k, v, heads, kv_div, TILED)


@pytest.mark.parametrize("dh", [40, 80, 160])
@pytest.mark.parametrize("L", [300, 129])
def test_tiled_kernel_qkv_column_slices(dh, L):
    """q, k and v as column slices of one [I, L, 3C] projection output (row stride 3C), as the spatial transformer passes them."""
    heads, images = 2, 3
    q, k, v = make_case("peaked", L, L, heads, dh, images=images, seed=dh + L, logit=30.0)
    qkv = torch.cat([q, k, v], -1).cuda()
    C = heads * dh
    o = _run(qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:], heads, 1, TILED).cpu()
    err = (o.double() - attention_fp64(q, k, v, heads)).abs().max().item()
    assert err <= tol_fp32(q, k, v, heads), err


@pytest.mark.parametrize("case", ["peaked60", "jump200@last", "jump40@last", "staircase", "descending", "offset200", "uniform"])
@pytest.mark.parametrize("Lq,Lkv,dh,kv_div", [(100, 300, 40, 1), (64, 257, 80, 1), (50, 130, 160, 1), (60, 77, 80, 2)])
def test_tiled_and_checker_side_by_side(case, Lq, Lkv, dh, kv_div):
    heads = 2
    q, k, v = make_case(Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, images=2 * kv_div, kv_div=kv_div, seed=7 * Lq + Lkv, **case_kw(case, Lkv))
    _check(q, k, v, heads, kv_div, TILED)
    _check(q, k, v, heads, kv_div, CHECKER)


def test_default_selection_on_both_sides_of_the_crossover():
    import neurons_b200 as nb
    for Lq, Lkv, dh, kernel in ((128, 255, 40, "checker"), (128, 256, 40, "tiled"), (100, 300, 80, "checker"), (2048, 2048, 80, "tiled")):
        heads, images = 2, 2
        assert (Lq * Lkv * heads * images >= F32_TILED_MIN_SCORES) == (kernel == "tiled")
        q, k, v = (t.cuda() for t in make_case("peaked", Lq, Lkv, heads, dh, images=images, logit=10.0))
        _assert_default_runs(kernel, q, k, v, heads)
    with pytest.raises(nb.NmmError):          # forcing the tiled kernel on operands it cannot stream is an error, not a silent fall-back
        q = torch.randn(2, 64, 2 * 40 + 1, device="cuda")[..., 1:]
        _run(q, q, q, 2, 1, TILED)


# ---- the UNet's full sizes through the default selection ---------------------------------------------------------------------------
@pytest.mark.parametrize("L,dh", [(4096, 40), (1024, 80)])
def test_full_size_default_selection(L, dh):
    """16 images x 8 heads (config 2's CFG batch 2 x 8 frames): 4096 keys at d_h 40 is the 64 x 64 level the checker refused (2.1e9 score
    elements).  Two (image, head) pairs are checked fully against fp64, every other pair on a sample of rows."""
    heads, images = 8, 16
    C = heads * dh
    g = torch.Generator().manual_seed(L + dh)
    qkv = torch.randn(images, L, 3 * C, generator=g)
    qkv[..., :C] *= 6.0                                   # max |logit| of about 30
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    qc = qkv.cuda()
    o = _assert_default_runs("tiled", qc[..., :C], qc[..., C:2 * C], qc[..., 2 * C:], heads).cpu()
    assert torch.isfinite(o).all()
    rows = torch.randperm(L, generator=g)[:24]
    for i in range(images):
        full = i in (0, images - 1)
        r = slice(None) if full else rows
        qi = q[i:i + 1, r]
        ref = attention_fp64(qi, k[i:i + 1], v[i:i + 1], heads)
        err = (o[i:i + 1, r].double() - ref).abs().max().item()
        tol = tol_fp32(qi, k[i:i + 1], v[i:i + 1], heads)
        assert err <= tol, (i, err, tol)


# ---- the spatial transformer in FMA mode ----------------------------------------------------------------------------------------------
def _mirror(cfg, params, fma):
    import neurons_b200 as nb
    m = nb.Transformer3DModel(num_attention_heads=cfg.heads, attention_head_dim=cfg.head_dim, in_channels=cfg.channels, num_layers=cfg.layers,
                              cross_attention_dim=cfg.ctx_dim, use_linear_projection=not cfg.conv_proj, unet_use_cross_frame_attention=False,
                              unet_use_temporal_attention=False)
    m.load_state_dict(params, strict=True)
    m = m.eval().cuda()
    if fma:
        m.__dict__["_nmm_fp32_fma"] = True
    return m


def _self_attention_max_logit(params, x_img, cfg):
    """max |q k^T| / sqrt(d_h) of attn1 on one [1, C, 1, H, W] image (attention.py:106-110, 260-262, in fp64)."""
    p = {n: t.double() for n, t in params.items()}
    C = cfg.channels
    hs = torch.nn.functional.group_norm(x_img[:, :, 0].double(), so.GN_GROUPS, p["norm.weight"], p["norm.bias"], so.GN_EPS)
    hs = torch.nn.functional.conv2d(hs, p["proj_in.weight"], p["proj_in.bias"]).flatten(2).transpose(1, 2)
    n = torch.nn.functional.layer_norm(hs, (C,), p["transformer_blocks.0.norm1.weight"], p["transformer_blocks.0.norm1.bias"], so.LN_EPS)
    q = (n @ p["transformer_blocks.0.attn1.to_q.weight"].T).view(-1, cfg.heads, C // cfg.heads).transpose(0, 1)
    k = (n @ p["transformer_blocks.0.attn1.to_k.weight"].T).view(-1, cfg.heads, C // cfg.heads).transpose(0, 1)
    return (q @ k.transpose(-1, -2)).abs().max().item() * (C // cfg.heads) ** -0.5


def _peaked_params(cfg, seed, x_img, logit):
    """so.make_params with to_q and to_k of attn1 scaled so that the self-attention's max |logit| on x_img is `logit`."""
    params = so.make_params(cfg, seed)
    f = math.sqrt(logit / _self_attention_max_logit(params, x_img, cfg))
    for n in ("to_q", "to_k"):
        params[f"transformer_blocks.0.attn1.{n}.weight"] = params[f"transformer_blocks.0.attn1.{n}.weight"] * f
    assert abs(_self_attention_max_logit(params, x_img, cfg) - logit) < 0.01 * logit
    return params


@pytest.mark.parametrize("logit", [30.0, 60.0])
@pytest.mark.parametrize("C,side,B,frames", [(320, 64, 2, 8), (320, 32, 2, 16)])
def test_fma_mode_full_size_peaked(C, side, B, frames, logit):
    """config 2's 64 x 64 level (C = 320, B = 2, F = 8: refused before the tiled kernel) and NEURONS' shape (F = 16, 32 x 32): one (b, f)
    image of the FMA-mode call against the oracle on that image alone in fp64, bar 1e-4.  The x3 mode's error on the same input is printed."""
    cfg = so.SpatialConfig(C, 8, 1, 768, True)
    x, ctx = so.make_inputs(cfg, B, frames, side, side, 77, 52)
    b, f = B - 1, frames // 2
    params = _peaked_params(cfg, 51, x[b:b + 1, :, f:f + 1], logit)
    ref = so.forward_reference_order({n: t.double() for n, t in params.items()}, x[b:b + 1, :, f:f + 1].double(), ctx[b:b + 1].double(), cfg)
    errs = {}
    with torch.no_grad():
        for fma in (True, False):
            y = _mirror(cfg, params, fma)(x.cuda(), encoder_hidden_states=ctx.cuda()).sample
            torch.cuda.synchronize()
            assert torch.isfinite(y).all()
            errs["fma" if fma else "x3"] = (y[b:b + 1, :, f:f + 1].double().cpu() - ref).abs().max().item()
            del y
    print(f"C={C} {side}x{side} B={B} F={frames} max|logit| {logit:g}: fma {errs['fma']:.2e}   x3 {errs['x3']:.2e} (x3 not asserted)")
    assert errs["fma"] <= TOL_FP32, errs


def test_fma_mode_graph_capture_above_the_crossover():
    """The FMA-mode call with the tiled kernel (2 images x 8 heads x 1024^2 score elements) captured in a CUDA graph and replayed on new data."""
    cfg = so.SpatialConfig(320, 8, 1, 768, True)
    x, ctx = so.make_inputs(cfg, 1, 2, 32, 32, 77, 61)
    assert 2 * 8 * 1024 * 1024 >= F32_TILED_MIN_SCORES
    params = _peaked_params(cfg, 60, x[:, :, 1:2], 40.0)
    m = _mirror(cfg, params, True)
    xs, cs = x.cuda(), ctx.cuda()
    with torch.no_grad():
        y_eager = m(xs, encoder_hidden_states=cs).sample.clone()
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            m(xs, encoder_hidden_states=cs)
            with torch.cuda.graph(g, stream=s):
                y_graph = m(xs, encoder_hidden_states=cs).sample
        torch.cuda.current_stream().wait_stream(s)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(y_graph, y_eager)
        x2, _ = so.make_inputs(cfg, 1, 2, 32, 32, 77, 62)
        xs.copy_(x2.cuda())
        g.replay()
        torch.cuda.synchronize()
    p64 = {n: t.double() for n, t in params.items()}
    for f in (0, 1):
        ref = so.forward_reference_order(p64, x2[:, :, f:f + 1].double(), ctx.double(), cfg)
        err = (y_graph[:, :, f:f + 1].double().cpu() - ref).abs().max().item()
        assert err <= TOL_FP32, (f, err)
