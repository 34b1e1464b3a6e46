"""The fp32-exact tensor-core mode (NMM_F32X6): fp32 operands as three bf16 planes (hi | mid | lo) and six MMAs per product.

CPU: the three-plane split reconstructs fp32 to 2^-24; a float emulation of the GEMM's k-block schedule (products of one K16 step summed
exactly, fp32 accumulation across steps) meets an fp32-grade bound from K = 320 to 5120, in the small-terms-first order the kernel uses,
while the large-terms-first order and the x3 schedule fail it; the mode selection (module flag `_nmm_fp32_exact`, env NMM_FP32_EXACT).
GPU: ops.linear(x6=True) for every epilogue against fp64 (within 2x the FMA GEMM's error), the x6 spatial attention against fp64 on every
edge-case kind of test_attention_edges.py (the fp32 kernels' bound), the module fixtures and the full-size peaked spatial shapes (within
2x the FMA mode's error and 1e-4), CUDA-graph capture, and the kernels an x6 call launches."""
import math

import pytest
import torch

from tests.helpers import TOL_FP32

# ---- float emulation of the tcgen05 k-block schedules (gemm_tcgen05.cu, PL) -------------------------------------------------------------
X6_ORDER = [(2, 0), (1, 1), (0, 2), (1, 0), (0, 1), (0, 0)]     # (A plane, W plane) per pass, small terms first: the kernel's order
X6_LARGE_FIRST = X6_ORDER[::-1]
X3_ORDER = [(0, 0), (0, 1), (1, 0)]                                 # the x3 kernel's order: hi.hi, hi.lo, lo.hi


def _planes(x, n):
    """fp32 -> n bf16 planes as float64 (hi = bf16(x), each next plane = bf16 of the fp32 remainder)."""
    r, out = x.float(), []
    for _ in range(n):
        p = r.to(torch.bfloat16)
        out.append(p.double())
        r = r - p.float()
    return out


def emulate_gemm(A, W, order, planes):
    """A [M, K] . W [N, K]^T as the tensor core runs it: per pass and K16 step the 16 plane products summed exactly (bf16 x bf16 is exact
    in fp32; summing them in fp64 leaves the one rounding per step), added to an fp32 accumulator."""
    a, w = _planes(A, planes), _planes(W, planes)
    M, K = A.shape
    N, nb = W.shape[0], K // 16
    acc = torch.zeros(M, N, dtype=torch.float32)
    for pa, pw in order:
        blk = torch.einsum("mbk,nbk->bmn", a[pa].view(M, nb, 16), w[pw].view(N, nb, 16))
        for b in range(nb):
            acc = (acc.double() + blk[b]).float()
    return acc.double()


def fp32_grade_bound(A, W):
    """Per output: 2^-24 * (2 S + 2 R), S = sqrt(sum_k (a_k w_k)^2) (the scale of the operand rounding, random in sign) and R = sqrt of the
    sum over K16 steps of the squared exact partial sums (the scale of the fp32 accumulator's roundings).  About seven standard deviations
    of an fp32-accumulated sum of exactly represented products."""
    prod = A.double().unsqueeze(1) * W.double().unsqueeze(0)
    M, N, K = prod.shape
    S = prod.pow(2).sum(-1).sqrt()
    R = prod.view(M, N, K // 16, 16).sum(-1).cumsum(-1).pow(2).sum(-1).sqrt()
    return prod.sum(-1), 2.0 ** -24 * (2.0 * S + 2.0 * R)


@pytest.mark.parametrize("kind", ["randn", "near_pow2", "large", "small"])
def test_three_plane_split_reconstructs_fp32(kind):
    from neurons_b200 import ops
    g = torch.Generator().manual_seed(3)
    x = torch.randn(64, 256, generator=g)
    if kind == "near_pow2":
        e = torch.randint(-20, 20, (64, 256), generator=g).float()
        x = torch.sign(x) * torch.exp2(e) * (1.0 + torch.randint(-3, 4, (64, 256), generator=g).float() * 2.0 ** -23)
    elif kind == "large":
        x = x * 1e30
    elif kind == "small":
        x = x * 1e-20          # the lo plane stays a normal number (|x| >= 2^-102); below that the split keeps what fp32 subnormals keep
    p = ops.split_planes(x, planes=3)
    assert p.dtype == torch.bfloat16 and p.shape == (64, 3 * 256)
    back = p[:, :256].double() + p[:, 256:512].double() + p[:, 512:].double()
    err = (back - x.double()).abs()
    assert (err <= 2.0 ** -24 * x.double().abs()).all(), (err / x.double().abs()).max().item()
    assert ((ops.merge_planes(p, 3).double() - x.double()).abs() <= 2.0 ** -23 * x.double().abs()).all()
    # the two-plane split is the x3 format, unchanged
    p2 = ops.split_planes(x)
    assert torch.equal(p2[:, :256], x.to(torch.bfloat16)) and torch.equal(p2[:, 256:], (x - x.to(torch.bfloat16).float()).to(torch.bfloat16))


@pytest.mark.parametrize("K", [320, 640, 1280, 2560, 5120])
def test_six_product_emulation_is_fp32_grade_and_x3_is_not(K):
    g = torch.Generator().manual_seed(K)
    A = torch.randn(32, K, generator=g)
    W = torch.randn(32, K, generator=g) / math.sqrt(K)
    ref, bound = fp32_grade_bound(A, W)
    r6 = ((emulate_gemm(A, W, X6_ORDER, 3) - ref).abs() / bound).max().item()
    r6l = ((emulate_gemm(A, W, X6_LARGE_FIRST, 3) - ref).abs() / bound).max().item()
    r3 = ((emulate_gemm(A, W, X3_ORDER, 2) - ref).abs() / bound).max().item()
    print(f"K={K}: max err / bound  x6 small-first {r6:.3f}   x6 large-first {r6l:.3f}   x3 {r3:.2f}")
    assert r6 <= 1.0, r6
    assert r3 >= 10.0, r3                  # the bound discriminates: the x3 schedule is not fp32-grade
    assert r6l > r6                        # the kernel's order (small terms first) is the more accurate one


# ---- mode selection ------------------------------------------------------------------------------------------------------------------
def _motion(C=320, heads=8):
    import neurons_b200 as nb
    return nb.get_motion_module(C, "Vanilla", dict(num_attention_heads=heads, num_transformer_block=1, temporal_position_encoding=True,
                                                   temporal_position_encoding_max_len=24, zero_initialize=False))


def _spatial(C=320, ctx_dim=768):
    import neurons_b200 as nb
    return nb.Transformer3DModel(num_attention_heads=8, attention_head_dim=C // 8, in_channels=C, num_layers=1, cross_attention_dim=ctx_dim)


@pytest.fixture
def no_mode_env(monkeypatch):
    from neurons_b200 import ops
    monkeypatch.setattr(ops, "_FP32_FMA_ENV", None)
    monkeypatch.setattr(ops, "_FP32_EXACT_ENV", None)
    return ops


def test_default_selection_is_unchanged_without_the_flag(no_mode_env):
    from neurons_b200 import lib as nlib
    from neurons_b200 import motion_module as mm
    from neurons_b200 import spatial_transformer as st
    ops = no_mode_env
    cfg = mm.config_of(_motion())
    assert not cfg.fp32_exact
    assert ops._dtype_code(torch.float32, cfg) == nlib.NMM_F32X3 and ops._dtype_code(torch.bfloat16, cfg) == nlib.NMM_BF16
    assert ops._dtype_code(torch.float32, mm.config_of(_motion(32, 8))) == nlib.NMM_F32
    m = _motion()
    m.__dict__["_nmm_fp32_fma"] = True
    assert ops._dtype_code(torch.float32, mm.config_of(m)) == nlib.NMM_F32
    scfg = st.spatial_config_of(_spatial())
    assert not scfg.fp32_exact and st._dtype_code(torch.float32, scfg) == nlib.NMM_F32X3


def test_exact_flag_selects_x6_for_fp32_with_64_aligned_widths(no_mode_env, monkeypatch):
    from neurons_b200 import lib as nlib
    from neurons_b200 import motion_module as mm
    from neurons_b200 import spatial_transformer as st
    ops = no_mode_env
    for C, want in ((320, nlib.NMM_F32X6), (640, nlib.NMM_F32X6), (32, nlib.NMM_F32), (96, nlib.NMM_F32)):
        m = _motion(C, 8 if C % 8 == 0 else 1)
        m.__dict__["_nmm_fp32_exact"] = True
        cfg = mm.config_of(m)
        assert ops._dtype_code(torch.float32, cfg) == want, C
        assert ops._dtype_code(torch.bfloat16, cfg) == nlib.NMM_BF16          # bf16 activations ignore the flag
    for C, D, want in ((320, 768, nlib.NMM_F32X6), (320, 96, nlib.NMM_F32), (1280, 1024, nlib.NMM_F32X6)):
        s = _spatial(C, D)
        s.__dict__["_nmm_fp32_exact"] = True
        cfg = st.spatial_config_of(s)
        assert st._dtype_code(torch.float32, cfg) == want, (C, D)
        assert st._dtype_code(torch.bfloat16, cfg) == nlib.NMM_BF16
    # the environment variable selects it for every module
    monkeypatch.setattr(ops, "_FP32_EXACT_ENV", "1")
    assert ops._dtype_code(torch.float32, mm.config_of(_motion())) == nlib.NMM_F32X6
    assert st._dtype_code(torch.float32, st.spatial_config_of(_spatial())) == nlib.NMM_F32X6


def test_exact_and_fma_together_raise(no_mode_env, monkeypatch):
    from neurons_b200 import motion_module as mm
    from neurons_b200 import spatial_transformer as st
    ops = no_mode_env
    for mod, cfg_of in ((_motion(), mm.config_of), (_spatial(), st.spatial_config_of)):
        mod.__dict__["_nmm_fp32_exact"] = True
        mod.__dict__["_nmm_fp32_fma"] = True
        with pytest.raises(ValueError, match="select one"):
            cfg_of(mod)
    m = _motion()
    m.__dict__["_nmm_fp32_fma"] = True
    monkeypatch.setattr(ops, "_FP32_EXACT_ENV", "1")
    with pytest.raises(ValueError, match="select one"):
        mm.config_of(m)
    monkeypatch.setattr(ops, "_FP32_EXACT_ENV", None)
    monkeypatch.setattr(ops, "_FP32_FMA_ENV", "1")
    m = _motion()
    m.__dict__["_nmm_fp32_exact"] = True
    with pytest.raises(ValueError, match="select one"):
        mm.config_of(m)


def test_exact_flag_is_part_of_the_packed_cache_key():
    from neurons_b200 import motion_module as mm
    m = _motion()
    before = mm._Engine._flags(m)
    m.__dict__["_nmm_fp32_exact"] = True
    assert mm._Engine._flags(m) != before


# ---- GPU ------------------------------------------------------------------------------------------------------------------------------
def _maxabs(a, b):
    return (a.double().cpu() - b.double().cpu()).abs().max().item()


def _gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


@pytest.mark.gpu
@pytest.mark.parametrize("epilogue", ["store", "residual", "residual_out", "geglu", "output"])
@pytest.mark.parametrize("K", [320, 640, 1280, 2560, 5120])
def test_linear_x6_vs_fp64(epilogue, K):
    """ops.linear(x6=True) against fp64 on every epilogue the mode takes: within 2x the FMA GEMM's (NMM_F32) error on the same inputs."""
    from neurons_b200 import lib as nlib
    from neurons_b200 import ops
    g = torch.Generator().manual_seed(K)
    M, N = 256, 640
    A = torch.randn(M, K, generator=g)
    Wt = torch.randn(N if epilogue != "output" else 320, K, generator=g) / math.sqrt(K)
    bias = 0.1 * torch.randn(Wt.shape[0], generator=g)
    acc = A.double() @ Wt.double().T + bias.double()
    Ad, Wd, bd = A.cuda(), Wt.cuda(), bias.cuda()
    errs = {}
    for mode in ("fma", "x6", "x3"):              # x3: printed for comparison, not asserted
        kw = dict(x6=(mode == "x6"), x3=(mode == "x3"))
        if epilogue == "store":
            h = torch.empty(M, N, device="cuda")
            ops.linear(Ad, Wd, bd, nlib.EPI_STORE, h=h, want_out=False, **kw)
            got, ref = h, acc
        elif epilogue in ("residual", "residual_out"):
            h0 = torch.randn(M, N, generator=g)
            h = h0.cuda()
            out = ops.linear(Ad, Wd, bd, nlib.EPI_RESIDUAL, h=h, want_out=epilogue == "residual_out", **kw)
            got, ref = (out if epilogue == "residual_out" else h), acc + h0.double()
            if epilogue == "residual_out":
                assert torch.equal(h.cpu(), h0)                 # h is only read
        elif epilogue == "geglu":
            got = ops.linear(Ad, Wd, bd, nlib.EPI_GEGLU, **kw)
            a4 = acc.view(M, N // 4, 4)
            ref = torch.stack([a4[..., 0] * _gelu64(a4[..., 2]), a4[..., 1] * _gelu64(a4[..., 3])], -1).reshape(M, N // 2)
        else:
            x = torch.randn(1, 320, 2, 8, 16, generator=g)
            cfg = ops.ModuleConfig(320)
            got = ops.linear(Ad, Wd, bd, nlib.EPI_OUTPUT, cfg=cfg, x=x.cuda(), **kw)
            ref = acc.reshape(1, 2, 128, 320).permute(0, 3, 1, 2).reshape(1, 320, 2, 8, 16) + x.double()
        torch.cuda.synchronize()
        assert got.dtype == torch.float32 and got.shape == ref.shape
        errs[mode] = _maxabs(got, ref)
    print(f"{epilogue} K={K}: fma {errs['fma']:.2e}  x6 {errs['x6']:.2e}  x3 {errs['x3']:.2e}")
    assert errs["x6"] <= 2.0 * errs["fma"], errs


def _x6_attention_params():
    from tests.test_attention_edges import cases
    shapes = [(100, 300, 40, 1), (257, 513, 80, 1), (130, 1024, 160, 1), (65, 33, 40, 1), (60, 77, 40, 2), (100, 77, 80, 8), (33, 77, 160, 2)]
    out = []
    for Lq, Lkv, dh, kv_div in shapes:
        kws = cases(Lkv) if (Lq, Lkv) == (100, 300) else cases(Lkv, jumps=(8.5, 40.0, 200.0), ats=("t1", "last") if Lkv > 128 else ())
        for cid, kw in kws:
            out.append(pytest.param(kw, Lq, Lkv, dh, kv_div, id=f"{cid}-Lq{Lq}-Lkv{Lkv}-dh{dh}-kvdiv{kv_div}"))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("kw,Lq,Lkv,dh,kv_div", _x6_attention_params())
def test_x6_attention_vs_fp64(kw, Lq, Lkv, dh, kv_div):
    """Peaked (max |logit| up to 60), jumps up to 200 log2 units, descending / underflow, row offsets, uniform rows over ragged tiles, the
    text cross-attention's kv_div: the bound the FMA-pipe kernels are held to (tol_fp32)."""
    import neurons_b200 as nb
    from tests.test_attention_edges import attention_fp64, make_case, tol_fp32
    heads = 2
    q, k, v = make_case(Lq=Lq, Lkv=Lkv, heads=heads, dh=dh, images=2 * kv_div, kv_div=kv_div, seed=Lq + Lkv + dh, **kw)
    o = nb.spatial_attention(q.cuda(), k.cuda(), v.cuda(), heads, kv_div, x6=True)
    torch.cuda.synchronize()
    assert o.dtype == torch.float32
    err = _maxabs(o, attention_fp64(q, k, v, heads, kv_div))
    tol = tol_fp32(q, k, v, heads, kv_div)
    assert math.isfinite(err) and err <= tol, (err, tol)


@pytest.mark.gpu
@pytest.mark.parametrize("name", __import__("tests.helpers", fromlist=["golden_names"]).golden_names())
def test_motion_module_golden_x6_vs_fp64(name):
    """Both exact modes within the fp32 bar of the fixture's fp32 reference output, and x6 within 2x the FMA mode's error against the
    oracle in fp64.  (Against the fp32 reference both errors are 1-2e-6, the size of that reference's own rounding: at c320_f8_8x8_a2 the
    x6 mode's worst element is 2.4e-6 from the fp32 reference, which is itself 1.4e-6 from fp64 there.)"""
    from oracle import motion_oracle as mo
    from tests import helpers
    fx, cfg, params, x = helpers.load_golden(name)
    ref64 = mo.forward_reference_order({k: v.double() for k, v in params.items()}, x.double(), cfg)
    errs, errs64 = {}, {}
    with torch.no_grad():
        for flag in ("_nmm_fp32_fma", "_nmm_fp32_exact"):
            m = helpers.mirror_module(cfg, params, "cuda")
            m.__dict__[flag] = True
            y = m(x.cuda(), None, None)
            errs[flag], errs64[flag] = _maxabs(y, fx["out_ref_fp32"]), _maxabs(y, ref64)
    print(name, errs, errs64)
    assert errs["_nmm_fp32_exact"] <= TOL_FP32 and errs["_nmm_fp32_fma"] <= TOL_FP32, errs
    assert errs64["_nmm_fp32_exact"] <= 2.0 * errs64["_nmm_fp32_fma"], errs64


def _sp_mirror(cfg, params, flag):
    import neurons_b200 as nb
    m = nb.Transformer3DModel(num_attention_heads=cfg.heads, attention_head_dim=cfg.head_dim, in_channels=cfg.channels, num_layers=cfg.layers,
                              cross_attention_dim=cfg.ctx_dim, use_linear_projection=not cfg.conv_proj, unet_use_cross_frame_attention=False,
                              unet_use_temporal_attention=False)
    m.load_state_dict(params, strict=True)
    m = m.eval().cuda()
    if flag:
        m.__dict__[flag] = True
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("name", __import__("tests.test_spatial_oracle", fromlist=["sp_golden_names"]).sp_golden_names())
def test_spatial_golden_x6(name):
    from tests.test_spatial_oracle import load_sp_golden
    fx, cfg, params, x, ctx = load_sp_golden(name)
    errs = {}
    with torch.no_grad():
        for flag in ("_nmm_fp32_fma", "_nmm_fp32_exact"):
            y = _sp_mirror(cfg, params, flag)(x.cuda(), encoder_hidden_states=ctx.cuda()).sample
            errs[flag] = _maxabs(y, fx["out_ref_fp32"])
    print(name, errs)
    assert errs["_nmm_fp32_exact"] <= TOL_FP32 and errs["_nmm_fp32_exact"] <= 2.0 * errs["_nmm_fp32_fma"], errs


@pytest.mark.gpu
@pytest.mark.parametrize("logit", [30.0, 60.0])
@pytest.mark.parametrize("C,side,B,frames", [(320, 64, 2, 8), (320, 32, 2, 16)])
def test_x6_mode_full_size_peaked(C, side, B, frames, logit):
    """The shapes of test_fma_mode_full_size_peaked: one (b, f) image against the fp64 oracle on that image alone; x6 within 2x the FMA
    mode's error (x3 printed for comparison)."""
    from oracle import spatial_oracle as so
    from tests.test_spatial_fp32_attention import _peaked_params
    cfg = so.SpatialConfig(C, 8, 1, 768, True)
    x, ctx = so.make_inputs(cfg, B, frames, side, side, 77, 52)
    b, f = B - 1, frames // 2
    params = _peaked_params(cfg, 51, x[b:b + 1, :, f:f + 1], logit)
    ref = so.forward_reference_order({n: t.double() for n, t in params.items()}, x[b:b + 1, :, f:f + 1].double(), ctx[b:b + 1].double(), cfg)
    errs = {}
    with torch.no_grad():
        for mode, flag in (("fma", "_nmm_fp32_fma"), ("x6", "_nmm_fp32_exact"), ("x3", None)):
            y = _sp_mirror(cfg, params, flag)(x.cuda(), encoder_hidden_states=ctx.cuda()).sample
            torch.cuda.synchronize()
            assert torch.isfinite(y).all()
            errs[mode] = _maxabs(y[b:b + 1, :, f:f + 1], ref)
            del y
    print(f"C={C} {side}x{side} B={B} F={frames} max|logit| {logit:g}: fma {errs['fma']:.2e}  x6 {errs['x6']:.2e}  x3 {errs['x3']:.2e}")
    assert errs["x6"] <= 2.0 * errs["fma"] and errs["x6"] <= TOL_FP32, errs


def _graph_replay(fn, inp, new):
    with torch.no_grad():
        eager = fn().clone()
        g = torch.cuda.CUDAGraph()
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fn()
            with torch.cuda.graph(g, stream=s):
                out = fn()
        torch.cuda.current_stream().wait_stream(s)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, eager)
        inp.copy_(new)
        g.replay()
        torch.cuda.synchronize()
    return out


@pytest.mark.gpu
def test_x6_graph_capture_spatial_full_size_and_motion_module():
    from oracle import spatial_oracle as so
    from tests import helpers
    # spatial transformer, 64 x 64 latent (the full-size level), 2 frames
    cfg = so.SpatialConfig(320, 8, 1, 768, True)
    params = so.make_params(cfg, 71)
    x, ctx = so.make_inputs(cfg, 1, 2, 64, 64, 77, 72)
    x2, _ = so.make_inputs(cfg, 1, 2, 64, 64, 77, 73)
    m = _sp_mirror(cfg, params, "_nmm_fp32_exact")
    xs, cs = x.cuda(), ctx.cuda()
    y = _graph_replay(lambda: m(xs, encoder_hidden_states=cs).sample, xs, x2.cuda())
    ref = so.forward_reference_order({n: t.double() for n, t in params.items()}, x2[:, :, 1:2].double(), ctx.double(), cfg)
    assert _maxabs(y[:, :, 1:2], ref) <= TOL_FP32
    # motion module
    fx, mcfg, mparams, mx = helpers.load_golden("c320_f8_8x8_a2")
    mm_ = helpers.mirror_module(mcfg, mparams, "cuda")
    mm_.__dict__["_nmm_fp32_exact"] = True
    xin = torch.zeros_like(mx).cuda()
    y = _graph_replay(lambda: mm_(xin, None, None), xin, mx.cuda())
    assert _maxabs(y, fx["out_ref_fp32"]) <= TOL_FP32


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with torch.no_grad():
        fn()
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
    return {e.key for e in prof.key_averages()}


@pytest.mark.gpu
def test_x6_call_launches_the_x6_kernels():
    """An x6 call runs the six-product GEMM and attention kernels and no FMA-pipe GEMM or fp32 attention kernel; the same module without the
    flag runs the x3 kernels (re-packed: the flag is part of the engine's key); in the motion module likewise."""
    from oracle import spatial_oracle as so
    from tests import helpers
    cfg = so.SpatialConfig(320, 8, 1, 768, True)
    params = so.make_params(cfg, 81)
    x, ctx = so.make_inputs(cfg, 1, 2, 32, 32, 77, 82)
    xs, cs = x.cuda(), ctx.cuda()
    m = _sp_mirror(cfg, params, "_nmm_fp32_exact")
    names = " ".join(_kernel_names(lambda: m(xs, encoder_hidden_states=cs)))
    if not names:
        pytest.skip("CUPTI delivered no kernel records in this process")
    assert "linear_tc_kernel<" in names and ", 3>" in names and "spatial_attention_x6_kernel<40>" in names, names
    assert "linear_fp32_fma" not in names and "spatial_attention_f32" not in names and "spatial_attention_x3" not in names, names
    del m.__dict__["_nmm_fp32_exact"]
    names = " ".join(_kernel_names(lambda: m(xs, encoder_hidden_states=cs)))
    assert "spatial_attention_x3_kernel<40>" in names and "spatial_attention_x6" not in names and ", 3>" not in names, names
    fx, mcfg, mparams, mx = helpers.load_golden("c320_f8_8x8_a2")
    mm_ = helpers.mirror_module(mcfg, mparams, "cuda")
    mm_.__dict__["_nmm_fp32_exact"] = True
    names = " ".join(_kernel_names(lambda: mm_(mx.cuda(), None, None)))
    assert ", 3>" in names and "linear_fp32_fma" not in names, names
