#!/usr/bin/env python
"""Error of the GroupNorm and LayerNorm kernels against fp64 as the offset of a group (row) over its spread grows, next to torch fp32 on the
same input and the ulp floor of tests/test_norm_edges.py (ulp(max |x| of the group) / sqrt(var + eps) * |gamma|; the tests assert
err <= 4 floor + 1e-6 (1 + |ref|); `/bound` is the worst err / that bound, <= 1 passes).  Inputs are that file's constructors:
  gn_tokens / inflated_gn   fp32 offset groups (mu / sigma = 0 ... 3000) at C = 320, 64 x 64 (one CTA per group) and C = 320, 128 x 128
                            (three splits per group)
  layernorm_pe              fp32 rows, C = 320 (vec kernel) and 96 (generic kernel)
  decoder GN                temporal attention of the video decoder on near-static frames (base ~ 4 N(0, 1) + delta N(0, 1), t = 6,
                            cpg = 1), whole-block error against the fp64 oracle (its GroupNorm is inside; torch column: n/a)
Prints the GPU's name and power limit first.  Development / profiles tool."""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import neurons_b200 as nb  # noqa: E402
from neurons_b200 import ops  # noqa: E402
from tests import test_norm_edges as tn  # noqa: E402

DEV = "cuda"


def gpu_info():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    return f"{name}, power limit {pl}"


def row(label, ratio, err, over, terr):
    t = f"{terr:10.2e}" if terr is not None else "       n/a"
    print(f"{label:34s} {ratio:>6g} {err:10.2e} {over:8.2f} {t}")


def over_floor(got, ref, floor):
    return ((got.double().cpu() - ref).abs() / (tn.K_FLOOR * floor + tn.BASE * (1 + ref.abs()))).max().item()


def groupnorm_rows(shape, label):
    B, C, F, H, W = shape
    w, b = tn.affine(C, C)
    for ratio in tn.RATIOS_F32:
        x = tn.offset_groups(shape, ratio, seed=ratio + H)
        ref = tn.groupnorm64(x, w, b, tn.GN_EPS_MODULE)
        floor = tn.groupnorm_floor(x, w, tn.GN_EPS_MODULE)
        terr = tn._torch_gn_err(x, w, b, tn.GN_EPS_MODULE, ref)
        xd = x.to(DEV)
        tok = ops.groupnorm_tokens(nb.ModuleConfig(C, heads=1, pos_enc=False), xd, w.to(DEV), b.to(DEV))
        tok = tok.view(B, F, H, W, C).permute(0, 4, 1, 2, 3)
        row(f"gn_tokens fp32 {label}", ratio, (tok.double().cpu() - ref).abs().max().item(), over_floor(tok, ref, floor.expand(x.shape)), terr)
        y = ops.inflated_groupnorm(xd, w.to(DEV), b.to(DEV), tn.GN_EPS_MODULE)
        row(f"inflated_gn fp32 {label}", ratio, (y.double().cpu() - ref).abs().max().item(), over_floor(y, ref, floor.expand(x.shape)), terr)


def layernorm_rows(C):
    B, F, H, W = 1, 8, 16, 16
    N = B * F * H * W
    w, b = tn.affine(C, 5)
    for ratio in (0, 10, 100, 300, 1000):
        h = tn.offset_rows(N, C, ratio, seed=C + ratio)
        ref = torch.nn.functional.layer_norm(h.double(), (C,), w.double(), b.double(), 1e-5)
        hd = h.double()
        floor = torch.from_numpy(tn.ulp32(hd.abs().amax(1, keepdim=True).numpy())) / torch.sqrt(hd.var(1, unbiased=False, keepdim=True) + 1e-5) * w.double().abs()
        out = ops.layernorm_pe(nb.ModuleConfig(C), (B, F, H, W), h.to(DEV), w.to(DEV), b.to(DEV), None, torch.float32)
        terr = (torch.nn.functional.layer_norm(h, (C,), w, b, 1e-5).double() - ref).abs().max().item()
        row(f"layernorm_pe fp32 C={C}", ratio, (out.double().cpu() - ref).abs().max().item(), over_floor(out, ref, floor), terr)


def decoder_rows():
    from oracle import decoder_oracle as do
    from neurons_b200 import video_decoder as vd
    from tests.test_video_decoder import FakeAttention
    C = 32
    cfg = do.DecoderAttnConfig(C)
    params = do.make_params(cfg, C)
    p64 = {k: v.double() for k, v in params.items()}
    attn = FakeAttention(cfg, params).cuda().eval()
    for delta in (1.0, 0.1, 3e-2, 1e-2, 1e-3):
        x = tn.near_static_video(1, 6, C, 28, delta, seed=1)
        with torch.no_grad():
            y = vd.temporal_attention_blend(x.cuda(), attn, torch.nn.Parameter(torch.tensor([0.0])).cuda(), 6)
        err = (y.double().cpu() - tn._decoder_fp64(p64, x, 0.0, 6, cfg)).abs().max().item()
        print(f"{'decoder block fp32 C=32 (cpg 1)':34s} {'d=' + format(delta, 'g'):>6s} {err:10.2e} {'':8s} {'n/a':>10s}")


def main():
    print(gpu_info())
    print(f"{'kernel':34s} {'mu/sd':>6s} {'max err':>10s} {'/bound':>8s} {'torch fp32':>10s}")
    with torch.no_grad():
        groupnorm_rows((1, 320, 2, 64, 64), "C=320 64x64")
        groupnorm_rows((1, 320, 1, 128, 128), "C=320 128x128")
        layernorm_rows(320)
        layernorm_rows(96)
        decoder_rows()


if __name__ == "__main__":
    main()
