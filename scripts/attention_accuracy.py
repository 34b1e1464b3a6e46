#!/usr/bin/env python
"""Max-abs error of the attention kernels against fp64 as the logits grow: the spatial kernels (bf16 tcgen05, fp32-grade x3, fp32-exact x6,
fp32 checker, fp32 tiled)
and the temporal attention (bf16, fp32), on randn q scaled to a given max |logit| (tests/test_attention_edges.py `peaked`), |v| ~ N(0, 1).
For x3 it also prints what an fp64 emulation of the kernel's own arithmetic predicts (split, 3 products, fp32 scores, split weights), and for
reference what fp32 torch on the host gives.  Prints the GPU's name and power limit first.  Development / profiles tool."""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import neurons_b200 as nb  # noqa: E402
from neurons_b200 import lib as nlib  # noqa: E402
from neurons_b200 import ops  # noqa: E402
from oracle import motion_oracle as mo  # noqa: E402
from tests import test_attention_edges as te  # noqa: E402

LOGITS = tuple(int(a) for a in sys.argv[1:]) or (1, 4, 10, 20, 30, 40, 60)


def err(a, b):
    return (a.double().cpu() - b.double().cpu()).abs().max().item()


def torch_fp32(q, k, v, heads, kv_div):
    qq, kk, vv = (te._heads(t, heads).float() for t in (q, k, v))
    kk, vv = kk.repeat_interleave(kv_div, 0), vv.repeat_interleave(kv_div, 0)
    return te._merge(torch.softmax(qq @ kk.transpose(-1, -2) * qq.shape[-1] ** -0.5, -1) @ vv)


def main():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                            timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        pl = "unknown"
    print(f"# {name}, power limit {pl}")
    print("# spatial: 2 images x 2 heads, Lq 256, Lkv 1024 (x3 / fp32: Lq 128), q = randn scaled to max |logit|, k, v = randn")
    print(f"{'dh':>4} {'max|logit|':>10} {'bf16 tc':>10} {'x3':>10} {'x3 emul.':>10} {'x6':>10} {'fp32 chk':>10} {'fp32 tiled':>10} {'torch fp32':>10}")
    for dh in (40, 80, 160):
        for L in LOGITS:
            q, k, v = te.make_case("peaked", 256, 1024, 2, dh, seed=dh + L, logit=float(L))
            qb, kb, vb = (te.round_bf16(t) for t in (q, k, v))
            o = nb.spatial_attention(qb.cuda().bfloat16(), kb.cuda().bfloat16(), vb.cuda().bfloat16(), 2)
            e_bf16 = err(o, te.attention_fp64(qb, kb, vb, 2))
            q, k, v = te.make_case("peaked", 128, 1024, 2, dh, seed=dh + L, logit=float(L))
            ref = te.attention_fp64(q, k, v, 2)
            e_x3 = err(nb.spatial_attention(q.cuda(), k.cuda(), v.cuda(), 2, x3=True), ref)
            e_emu = err(te.x3_emulation(q, k, v, 2), ref)
            e_x6 = err(nb.spatial_attention(q.cuda(), k.cuda(), v.cuda(), 2, x6=True), ref)
            with nlib.options({nlib.OPT_SPATIAL_ATTN: 31}):          # NMM_F32: force the checker / the tiled kernel
                e_f32 = err(nb.spatial_attention(q.cuda(), k.cuda(), v.cuda(), 2), ref)
            with nlib.options({nlib.OPT_SPATIAL_ATTN: 30}):
                e_tiled = err(nb.spatial_attention(q.cuda(), k.cuda(), v.cuda(), 2), ref)
            e_t = err(torch_fp32(q, k, v, 2, 1), ref)
            print(f"{dh:>4} {L:>10} {e_bf16:>10.2e} {e_x3:>10.2e} {e_emu:>10.2e} {e_x6:>10.2e} {e_f32:>10.2e} {e_tiled:>10.2e} {e_t:>10.2e}", flush=True)
    print("# temporal: B 1, 3 x 3 positions, 8 heads; qkv randn with q scaled to max |logit|; kernel of NMM_OPT_ATTN_VARIANT 0")
    print(f"{'C':>5} {'F':>3} {'max|logit|':>10} {'bf16':>10} {'fp32':>10}")
    for C, F in ((320, 16), (1280, 24)):
        c = mo.MotionConfig(C, max_len=32)
        cfg = nb.ModuleConfig(c.channels, c.heads, c.layers, c.attn_blocks, c.pos_enc, c.max_len)
        for L in LOGITS:
            qkv = te._temporal_case(f"peaked{L}", F, C, 8, 9, seed=C + L)
            row = []
            for dt in (torch.bfloat16, torch.float32):
                x = te.round_bf16(qkv) if dt == torch.bfloat16 else qkv
                row.append(err(ops.temporal_attention(cfg, (1, F, 3, 3), x.cuda().to(dt)), te._temporal_fp64(x, 1, F, 9, 8)))
            print(f"{C:>5} {F:>3} {L:>10} {row[0]:>10.2e} {row[1]:>10.2e}", flush=True)


if __name__ == "__main__":
    main()
