#!/usr/bin/env python
"""bench.py -- motion-module throughput of one UNet denoising step (BASELINE.json config 2) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes the 20 module outputs of the last timed step (rank 0) as DIR/<call>.npy, float32: a fixed sample of
DUMP_ELEMS elements of each output's logical [B,C,F,H,W] order, the positions seeded by the output's size. The inputs come from a
generator of their own and the weights from name-keyed seeds (oracle.motion_oracle.make_params), so they do not depend on how a
build constructs its modules: two builds run with the same arguments can be compared output for output.

A "step" = the 20 motion-module calls of one UNet3DConditionModel.forward at SD1.5 512x512 (64x64 latent), 8 frames,
CFG batch 2, bf16 -- 20 distinct modules (417 M parameters), 20 distinct [2,C,8,L,L] activations in the
[B,F,C,H,W]-storage layout the UNet hands over.  Per step the inputs + weights touched (1.2 GB) exceed the 126 MB L2.
    value   motion-module TFLOP/s, algorithmic FLOPs (SURVEY 8(d)) / device time, inputs resident in HBM
    e2e     same metric through the public module call with HOST buffers: pinned H2D of every input and D2H of every
            output inside the timed region (copies pipelined against compute on separate streams); two regions of exactly K
            steps are timed, the better one is the value and both are listed (host-fabric noise on shared boxes)
    roofline  the dominant kernel (tcgen05 bf16 GEMM): algorithmic FLOPs of its launches / their summed device time,
            measured with CUDA events the library records around each launch on the launch stream
    cpu_baseline  the oracle port of the reference module (oracle/motion_oracle.py) timed on the host cores
    spatial_transformer  secondary (SURVEY 8(f) N3): the 16 spatial Transformer3DModel calls of the same UNet step, with the
            per-kernel split and stock torch eager on the same GPU;  clips: the 25-step clip loop (configs 2 / 3)
Each rank runs a full replica (weak scaling, no collective on the path); time = max over ranks.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LATENT, FRAMES, BATCH = 64, 8, 2
METRIC, UNIT = "motion-module fwd TFLOP/s", "TFLOP/s"
DUMP_ELEMS = 1 << 19          # per output: 20 x 2 MiB of float32, under 64 MB in all


def workload_config(n_gpus):
    return {"workload": "UNet3DConditionModel one denoising step, all 20 motion modules, SD1.5 512x512 (64x64 latent), 8 frames, CFG batch 2",
            "baseline_config": "configs[1]", "latent": LATENT, "frames": FRAMES, "batch": BATCH, "calls_per_step": 20,
            "layout": "[B,F,C,H,W]-storage views (UNet call sites)", "parallelism": f"dp{n_gpus} replicas, no collective on the path",
            "l2": "inputs larger than L2: 20 distinct activations + 20 modules' weights = 1.2 GB per step vs 126 MB L2"}


# ---------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms during the timed region (B200_PROFILING.md)."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.rows = []
        self.proc = None
        self.thread = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) >= 8 and parts[0].isdigit() and int(parts[0]) == self.gpu_index:
                self.rows.append(parts)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows for n, v in zip(names, r[4:8]) if v.lower().startswith("active")})
        pw = [float(r[3]) for r in self.rows if r[3].replace(".", "").isdigit()]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows), "power_w_max": max(pw) if pw else None}


def physical_gpu_index(local_rank: int) -> int:
    vis = os.environ.get("CUDA_VISIBLE_DEVICES")
    if vis:
        ids = [v for v in vis.split(",") if v.strip() != ""]
        if local_rank < len(ids) and ids[local_rank].strip().isdigit():
            return int(ids[local_rank])
    return local_rank


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_tflops": p.get("bf16_tflops"), "bf16_tflops_sustained": p.get("bf16_tflops_sustained"),
                "hbm_gbs": p.get("hbm_gbs"), "source": "measured (MEASURED_PEAKS.json)"}
    return {"bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "hbm_gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


def dump_positions(calls):
    """{output size: DUMP_ELEMS sorted positions in the logical [B,C,F,H,W] order}, seeded by the size alone, so that the sample is
    the same in every run and every build."""
    positions = {}
    for c in calls:
        n = BATCH * c.channels * FRAMES * c.side * c.side
        if n not in positions:
            positions[n] = torch.randperm(n, generator=torch.Generator().manual_seed(n))[:DUMP_ELEMS].sort().values
    return positions


# ---------------------------------------------------------------------------------------------------------------
def clip_loop(nb, wl, dev, clips: int = 3, clip_batch: int = 1):
    """Second half of BASELINE.json's metric: 25-step clips/s at the NEURONS 'enhance' shape (configs[2]: CFG batch 2, 16 frames,
    256x256 video = 32x32 latent) -- the motion modules ONLY (20 UNet + 8 SparseCtrl-ControlNet calls per denoising step,
    scripts/neuroclips_video_enhance.py:356-358, pipeline_neuroclips.py:433-483); the rest of the UNet is outside the path.
    One step is captured in a CUDA graph and replayed 25 times per clip.  Returns (ms per clip on this rank, flops per clip)."""
    F, L, B, steps = 16, 32, 2 * clip_batch, 25              # CFG doubles the batch (pipeline_neuroclips.py:435)
    calls = wl.unet_step_calls(L) + wl.controlnet_step_calls(L)
    mods, xs = [], []
    with torch.no_grad():
        for c in calls:
            kw = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=("Temporal_Self",) * c.attn_blocks,
                      temporal_position_encoding=True, temporal_position_encoding_max_len=c.max_len, temporal_attention_dim_div=1,
                      zero_initialize=False)
            with torch.device(dev):
                mods.append(nb.get_motion_module(c.channels, "Vanilla", kw).to(torch.bfloat16).eval())
            xs.append(torch.randn(B, F, c.channels, c.side, c.side, device=dev, dtype=torch.bfloat16).permute(0, 2, 1, 3, 4))

        def one_step():
            for m, x in zip(mods, xs):
                m(x, None, None)

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            for _ in range(2):
                one_step()
            side.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                one_step()
        torch.cuda.current_stream().wait_stream(side)
        for _ in range(steps):
            graph.replay()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(clips * steps):
            graph.replay()
        e1.record()
        torch.cuda.synchronize()
    flops_clip = steps * sum(wl.module_flops(c.channels, B * F * c.side * c.side, F, c.attn_blocks) for c in calls)
    return e0.elapsed_time(e1) / clips, flops_clip           # ms per replayed 25-step loop (= clip_batch clips), flops of that loop


def clip_e2e(nb, wl, dev, rank: int, world: int, clips_per_rank: int = 4):
    """Clip-level end to end (BASELINE configs[2] shape), everything inside the timed region: per clip the H2D copy of its latents +
    conditioning from pinned host memory, 25 graph-replayed denoising steps (28 motion-module calls + the fused CFG / DDIM update,
    nmm_cfg_ddim_step, on the clip's latents), a decoded-frame-sized result per clip ([3, 16, 256, 256] fp16; nearest up-sampling stands
    for the VAE, which is outside the path) copied D2H, and -- once, at the end -- the gather of every rank's frames over NCCL
    (neurons_b200.sharding.gather_clips: the only collective of the path).  Clips are assigned round-robin exactly like the reference.
    Returns (seconds for this rank's clips incl. the gather, clips on this rank, bytes H2D per clip, bytes D2H per clip)."""
    import torch.distributed as dist
    from neurons_b200 import ops, sampler, sharding
    F, L, steps = 16, 32, 25
    calls = wl.unet_step_calls(L) + wl.controlnet_step_calls(L)
    num_clips = clips_per_rank * world
    mine = sharding.shard_indices(num_clips, rank, world)
    sch = sampler.DDIMSchedule()
    ts = sch.timesteps(steps)
    with torch.no_grad():
        mods, xs = [], []
        for c in calls:
            kw = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=("Temporal_Self",) * c.attn_blocks,
                      temporal_position_encoding=True, temporal_position_encoding_max_len=c.max_len, temporal_attention_dim_div=1,
                      zero_initialize=False)
            with torch.device(dev):
                mods.append(nb.get_motion_module(c.channels, "Vanilla", kw).to(torch.bfloat16).eval())
            xs.append(torch.randn(2, F, c.channels, c.side, c.side, device=dev, dtype=torch.bfloat16).permute(0, 2, 1, 3, 4))
        lat = torch.zeros(1, 4, F, L, L, device=dev, dtype=torch.bfloat16)
        cond = torch.zeros(1, 4, 1, L, L, device=dev, dtype=torch.bfloat16)
        host_lat = [torch.randn(1, 4, F, L, L).to(torch.bfloat16).pin_memory() for _ in mine]
        host_cond = [torch.randn(1, 4, 1, L, L).to(torch.bfloat16).pin_memory() for _ in mine]
        host_frames = [torch.empty(3, F, 8 * L, 8 * L, dtype=torch.float16).pin_memory() for _ in mine]
        frames_dev = torch.empty(len(mine), 3, F, 8 * L, 8 * L, device=dev, dtype=torch.float16)
        eps_u = torch.empty_like(lat)
        eps_c = torch.empty_like(lat)

        def one_step_modules():
            y = None
            for i, (m, x) in enumerate(zip(mods, xs)):
                out = m(x, None, None)
                if i == 19:                                   # the UNet's last motion-module call: 320 channels at the full latent resolution
                    y = out
            # the step's noise prediction for the clip: 4 channels of that output, CFG pair (uncond | cond)
            eps_u.copy_(y[0:1, :4]); eps_c.copy_(y[1:2, :4])

        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            one_step_modules()
            side.synchronize()
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph, stream=side):
                one_step_modules()
        torch.cuda.current_stream().wait_stream(side)

        def run_clip(k):
            lat.copy_(host_lat[k], non_blocking=True)
            cond.copy_(host_cond[k], non_blocking=True)
            for t in ts:
                graph.replay()
                a_t, a_prev = sch.alphas(t, steps)
                ops.cfg_ddim_step(lat, eps_u, eps_c, 8.5, a_t, a_prev)
            fr = torch.nn.functional.interpolate(lat[0, :3].float(), scale_factor=8, mode="nearest").to(torch.float16)      # [3, F, 256, 256]
            frames_dev[k].copy_(fr)
            host_frames[k].copy_(fr, non_blocking=True)

        run_clip(0)                                         # warm-up (also of the NCCL communicator: its lazy initialisation is not the path)
        if world > 1:
            sharding.gather_clips(frames_dev, num_clips)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for k in range(len(mine)):
            run_clip(k)
        out = sharding.gather_clips(frames_dev, num_clips) if world > 1 else frames_dev
        torch.cuda.synchronize()
        secs = time.perf_counter() - t0
        assert rank != 0 or out.shape[0] == num_clips
    h2d = host_lat[0].numel() * 2 + host_cond[0].numel() * 2
    d2h = host_frames[0].numel() * 2
    return secs, len(mine), h2d, d2h


def cpu_reference_time(sample: str, threads: int):
    """Time the oracle port of the reference module (fp32, torch CPU, all host threads) on a bounded sample.
    Returns (tflops, seconds, description).  This is the ONE place bench.py executes oracle/ (as the baseline)."""
    from neurons_b200 import workloads as wl
    from oracle import motion_oracle as mo
    torch.set_num_threads(threads)
    calls = wl.unet_step_calls(LATENT)
    if sample == "step":
        chosen, desc = calls, "one full step: all 20 calls"
    elif sample == "shapes":
        seen, chosen = set(), []
        for c in calls:
            if (c.channels, c.side) not in seen:
                seen.add((c.channels, c.side)); chosen.append(c)
        desc = "one call per distinct (channels, latent) of the step: (320,64) (640,32) (1280,16) (1280,8), batch 2, 8 frames"
    else:
        chosen, desc = [calls[0]], "one (320 ch, 64x64) call of the step, batch 2, 8 frames"
    params = {}
    for c in chosen:
        if c.channels not in params:
            cfg = mo.MotionConfig(c.channels, 8, 1, c.attn_blocks, True, c.max_len)
            g = torch.Generator().manual_seed(c.channels)
            params[c.channels] = (cfg, {k: (torch.rand(s, generator=g) * 2 - 1) / (s[-1] ** 0.5 if len(s) == 2 else 1.0)
                                        for k, s in mo.param_shapes(cfg).items()})
    xs = {}
    for c in chosen:
        key = (c.channels, c.side)
        if key not in xs:
            xs[key] = mo.make_input((BATCH, c.channels, FRAMES, c.side, c.side), 1, layout="bfchw")
    flops = wl.step_flops(chosen, BATCH, FRAMES)

    def run():
        t0 = time.perf_counter()
        with torch.no_grad():
            for c in chosen:
                cfg, p = params[c.channels]
                mo.forward_reference_order(p, xs[(c.channels, c.side)], cfg)
        return time.perf_counter() - t0
    return flops, run, desc


def gpu_eager_baseline(dev, steps: int = 3):
    """The reference's op sequence (oracle port, op-for-op the reference's torch calls incl. its layout copies) on CUDA tensors under
    stock torch eager -- "the reference on the same box": what cuBLAS + ATen make of the same step, in bf16 and in fp32 (TF32 off).
    A reported anchor, not the product path.  Returns {dtype: {ms_per_step, tflops}}."""
    from neurons_b200 import workloads as wl
    from oracle import motion_oracle as mo
    calls = wl.unet_step_calls(LATENT)
    flops = wl.step_flops(calls, BATCH, FRAMES)
    out = {}
    tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        for dt in (torch.bfloat16, torch.float32):
            params, xs = {}, []
            g = torch.Generator().manual_seed(7)
            for c in calls:
                if c.channels not in params:
                    cfg = mo.MotionConfig(c.channels, 8, 1, c.attn_blocks, True, c.max_len)
                    params[c.channels] = (cfg, {k: ((torch.rand(s, generator=g) * 2 - 1) / (s[-1] ** 0.5 if len(s) == 2 else 1.0)).to(dev, dt)
                                                for k, s in mo.param_shapes(cfg).items()})
                xs.append(torch.randn(BATCH, FRAMES, c.channels, c.side, c.side, device=dev, dtype=dt).permute(0, 2, 1, 3, 4))

            def step():
                for c, x in zip(calls, xs):
                    cfg, prm = params[c.channels]
                    mo.forward_reference_order(prm, x, cfg)
            with torch.no_grad():
                step()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    step()
                e1.record()
                torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / steps
            out["bf16" if dt == torch.bfloat16 else "f32"] = {"ms_per_step": ms, "tflops": flops / (ms * 1e-3) / 1e12}
            del params, xs
            torch.cuda.empty_cache()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = tf32
    return out


def spatial_leg(nb, nlib, dev, steps: int = 5, eager: bool = True):
    """SURVEY 8(f) N3, the motion module's neighbour: the 16 spatial Transformer3DModel calls of the SAME UNet step (config 2: CFG batch 2,
    8 frames, 64 x 64 latent, bf16; 2 down + 3 up calls per CrossAttn level + the mid block, unet.py:157-258), device-resident, with the
    per-kernel split (second pass, CUDA-event pairs) and stock torch eager on the same GPU for the same calls.  Secondary metric."""
    from oracle import spatial_oracle as so          # flop count + the eager anchor's op sequence only; never the product path
    levels = [(320, LATENT, 5), (640, LATENT // 2, 5), (1280, LATENT // 4, 5), (1280, LATENT // 8, 1)]
    mods, xs, cfgs = [], [], []
    ctx = torch.randn(BATCH, 77, 768, device=dev, dtype=torch.bfloat16)
    flops = 0.0
    for C, side, n in levels:
        cfg = so.SpatialConfig(C, 8, 1, 768, True)
        for _ in range(n):
            with torch.device(dev):
                m = nb.Transformer3DModel(num_attention_heads=8, attention_head_dim=C // 8, in_channels=C, cross_attention_dim=768,
                                          unet_use_cross_frame_attention=False, unet_use_temporal_attention=False)
            mods.append(m.to(torch.bfloat16).eval())
            xs.append(torch.randn(BATCH, C, FRAMES, side, side, device=dev, dtype=torch.bfloat16))
            cfgs.append(cfg)
            flops += so.flops(cfg, BATCH, FRAMES, side * side, 77)

    def step():
        for m, x in zip(mods, xs):
            m(x, encoder_hidden_states=ctx)

    def timed(fn, k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k
    with torch.no_grad():
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        n0 = nb.launch_count()
        ms = timed(step, steps)
        launches = nb.launch_count() - n0
        nlib.profile_begin()
        for _ in range(steps):
            step()
        prof = nlib.profile_end()
        out = {"workload": "the 16 spatial Transformer3DModel calls of the same UNet step (GroupNorm, 1x1 proj_in, self-attention over h*w, "
                           "77-token text cross-attention, GEGLU FF, proj_out + residual); inputs larger than L2 (16 distinct activations + weights)",
               "ms_per_step": ms, "tflops": flops / (ms * 1e-3) / 1e12, "flops_per_step": flops, "gpu_launches": int(launches),
               "kernels": {k: {"launches": v["launches"], "ms_per_step": v["total_ms"] / steps,
                               "tflops": v["flops"] / (v["total_ms"] * 1e-3) / 1e12 if v["total_ms"] > 0 and v["flops"] > 0 else None}
                           for k, v in prof.items() if v["launches"]}}
        if eager:
            try:
                prm = [{k: v.detach() for k, v in m.state_dict().items()} for m in mods]

                def eager_step():
                    for p, x, cfg in zip(prm, xs, cfgs):
                        so.forward_reference_order(p, x, ctx, cfg)
                eager_step()
                torch.cuda.synchronize()
                ems = timed(eager_step, 2)
                out["gpu_eager_baseline"] = {"ms_per_step": ems, "tflops": flops / (ems * 1e-3) / 1e12,
                                             "note": "the reference's op sequence (materialised scores) under stock torch eager, bf16, same GPU"}
            except Exception as e:
                out["gpu_eager_baseline"] = {"error": repr(e)[:200]}
    del mods, xs
    torch.cuda.empty_cache()
    return out


def run_reference_arm(args, rank):
    """--impl reference: the reference's own CPU implementation of the path (oracle port; the reference is pure Python
    and ships no installable package), all host threads, same metric/config.  Rank 0 only."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    # size the per-step sample so that (steps + warmup) steps end within ~150 s
    flops1, run1, _ = cpu_reference_time("one", threads)
    t_probe = min(run1(), run1())
    rate = flops1 / t_probe
    from neurons_b200 import workloads as wl
    calls = wl.unet_step_calls(LATENT)
    total_steps = args.steps + args.warmup
    est_step = wl.step_flops(calls, BATCH, FRAMES) / rate
    est_shapes = est_step / 5.0
    sample = "step" if est_step * total_steps <= 150 else ("shapes" if est_shapes * total_steps <= 150 else "one")
    flops, run, desc = cpu_reference_time(sample, threads)
    for _ in range(args.warmup):
        run()
    times = [run() for _ in range(args.steps)]
    ms = 1e3 * sum(times) / len(times)
    val = flops / (ms * 1e-3) / 1e12
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args.gpus),
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the host-CPU baseline leg")
    ap.add_argument("--no-clips", action="store_true", help="skip the 25-step clip loop (secondary metric)")
    ap.add_argument("--no-eager", action="store_true", help="skip the stock-torch-eager GPU anchor")
    ap.add_argument("--no-spatial", action="store_true", help="skip the spatial-transformer leg (SURVEY 8(f) N3, secondary metric)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a fixed sample of the last timed step's outputs to DIR/<call>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours only")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import torch.distributed as dist
    import neurons_b200 as nb
    from neurons_b200 import lib as nlib
    from neurons_b200 import workloads as wl

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the motion-module path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    calls = wl.unet_step_calls(LATENT)
    flops_step = wl.step_flops(calls, BATCH, FRAMES)
    kwargs = dict(num_attention_heads=8, num_transformer_block=1, attention_block_types=("Temporal_Self", "Temporal_Self"),
                  temporal_position_encoding=True, temporal_position_encoding_max_len=24, temporal_attention_dim_div=1,
                  zero_initialize=False)      # random-init weights of the v3 architecture; proj_out NOT zeroed (else identity)
    from oracle import motion_oracle as mo          # seeded weights only; never the product path
    seed = 1234 + rank
    torch.manual_seed(seed)
    gen = torch.Generator(device=dev).manual_seed(seed)
    modules, xs_dev, xs_host, ys_host = [], [], [], []
    with torch.no_grad():
        for i, c in enumerate(calls):
            with torch.device(dev):
                m = nb.get_motion_module(c.channels, "Vanilla", kwargs)
            m.load_state_dict(mo.make_params(mo.MotionConfig(c.channels, 8, 1, c.attn_blocks, True, c.max_len), seed * 64 + i))
            modules.append(m.to(torch.bfloat16).eval())
            x = torch.randn(BATCH, FRAMES, c.channels, c.side, c.side, device=dev, dtype=torch.bfloat16, generator=gen).permute(0, 2, 1, 3, 4)
            xs_dev.append(x)
            xs_host.append(torch.empty((BATCH, FRAMES, c.channels, c.side, c.side), dtype=torch.bfloat16).pin_memory())
            xs_host[-1].copy_(x.permute(0, 2, 1, 3, 4))
            ys_host.append(torch.empty((BATCH, FRAMES, c.channels, c.side, c.side), dtype=torch.bfloat16).pin_memory())
    h2d_bytes = sum(t.numel() * 2 for t in xs_host)
    d2h_bytes = sum(t.numel() * 2 for t in ys_host)

    def step_resident(keep=False):
        # an output is dropped as soon as the next call is issued (its buffer then takes the next output, as in a UNet that consumes
        # it right away); keep=True returns them instead
        ys = []
        for m, x in zip(modules, xs_dev):
            y = m(x, None, None)
            if keep:
                ys.append(y)
        return ys

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad():
        # ---------------- device-resident arm ("value") ----------------
        # --dump-outputs: the last step of each loop keeps its outputs, the warm-up's so that the allocator already holds 20 output
        # buffers when the timed region reaches its own last step, the one that is written
        positions = {n: p.to(dev) for n, p in dump_positions(calls).items()} if args.dump_outputs else None
        for i in range(args.warmup):
            step_resident(keep=positions is not None and i == args.warmup - 1)
        barrier()
        sampler = ClockSampler(physical_gpu_index(local_rank))
        sampler.start()
        launches0 = nb.launch_count()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for i in range(args.steps):
            ys = step_resident(keep=positions is not None and i == args.steps - 1)
        ev1.record()
        barrier()
        ms_total = ev0.elapsed_time(ev1)
        launches = nb.launch_count() - launches0
        # sampled on the device at once, so that the outputs do not outlive the timed region
        dumped = [y.reshape(-1).index_select(0, positions[y.numel()]).float().cpu().numpy() for y in ys] if positions else None
        del ys
        # ---------------- same K steps again with the library's per-kernel CUDA events (roofline of the dominant kernel) --------
        # (kept out of the `value` region: an event between two kernels defeats programmatic dependent launch)
        nlib.profile_begin()
        ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev2.record()
        for _ in range(args.steps):
            step_resident()
        ev3.record()
        barrier()
        ms_profiled = ev2.elapsed_time(ev3)
        prof = nlib.profile_end()
        clocks = sampler.stop()

        # ---------------- end-to-end arm: host buffers, copies inside the timed region ----------------
        s_in, s_out, s_c = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.current_stream()
        x_stage = [torch.empty_like(x.permute(0, 2, 1, 3, 4).contiguous()) for x in xs_dev]     # [B,F,C,H,W] device staging
        ev_in = [torch.cuda.Event() for _ in calls]
        ev_c = [torch.cuda.Event() for _ in calls]

        def step_e2e():
            for i, m in enumerate(modules):
                with torch.cuda.stream(s_in):
                    s_in.wait_event(ev_c[i])                       # previous step's compute on this staging buffer is done
                    x_stage[i].copy_(xs_host[i], non_blocking=True)
                    ev_in[i].record(s_in)
                s_c.wait_event(ev_in[i])
                y = m(x_stage[i].permute(0, 2, 1, 3, 4), None, None)
                ev_c[i].record(s_c)
                with torch.cuda.stream(s_out):
                    s_out.wait_event(ev_c[i])
                    ys_host[i].copy_(y.permute(0, 2, 1, 3, 4), non_blocking=True)
                    y.record_stream(s_out)

        for _ in range(2):
            step_e2e()
        # two timed regions of exactly K steps each; the better one is reported and both are listed (`e2e.runs_ms_per_step`): the arm
        # depends on the host's PCIe / memory fabric, which these shared boxes occasionally disturb by 2-3x for a fraction of a second
        e2e_runs = []
        for _ in range(2):
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                step_e2e()
            torch.cuda.synchronize()
            e2e_runs.append(1e3 * (time.perf_counter() - t0) / args.steps)
        e2e_ms = min(e2e_runs)

        # the same host<->device traffic with no compute: the PCIe floor of the e2e arm (both directions concurrently)
        def step_copies():
            for i in range(len(modules)):
                with torch.cuda.stream(s_in):
                    x_stage[i].copy_(xs_host[i], non_blocking=True)
                with torch.cuda.stream(s_out):
                    ys_host[i].copy_(x_stage[i], non_blocking=True)
        step_copies()
        torch.cuda.synchronize()
        barrier()          # every rank copies at the same time: the floor must see the same host-fabric contention as the e2e arm does
        t0 = time.perf_counter()
        for _ in range(3):
            step_copies()
        torch.cuda.synchronize()
        copy_ms = 1e3 * (time.perf_counter() - t0) / 3
        barrier()

    eager = None
    if rank == 0 and not args.no_eager:
        try:
            eager = gpu_eager_baseline(dev)
        except Exception as e:        # a reported anchor only: never fail the bench line over it
            eager = {"error": repr(e)[:200]}
    spatial = None
    if rank == 0 and not args.no_spatial:
        try:
            spatial = spatial_leg(nb, nlib, dev, eager=not args.no_eager)
        except Exception as e:        # secondary metric: never fail the bench line over it
            spatial = {"error": repr(e)[:200]}
    clip_ms, clip_flops = (0.0, 0.0) if args.no_clips else clip_loop(nb, wl, dev)
    clip4_ms, clip4_flops = (0.0, 0.0) if args.no_clips else clip_loop(nb, wl, dev, clips=2, clip_batch=4)       # BASELINE configs[3]: 4 clips per GPU
    ce_secs, ce_n, ce_h2d, ce_d2h = (0.0, 0, 0, 0) if args.no_clips else clip_e2e(nb, wl, dev, rank, world)
    # max over ranks
    t = torch.tensor([ms_total, e2e_ms, clip_ms, clip4_ms, ce_secs, copy_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, clip_ms, clip4_ms, ce_secs, copy_ms = (float(v) for v in t)
    ms_step = ms_total / args.steps
    value = world * flops_step / (ms_step * 1e-3) / 1e12
    e2e_value = world * flops_step / (e2e_ms * 1e-3) / 1e12

    if rank == 0:
        peaks = measured_peaks()
        gemm, fused = prof["linear_bf16_tcgen05"], prof["fused_module_tcgen05"]
        # Denominator: the BURST cuBLAS figure.  The timed region is a fraction of a second at ~max SM clock (see `clocks`); the
        # sustained figure belongs to seconds-long loops under the power cap.  Both fractions are printed.
        peak_tf = peaks["bf16_tflops"] or peaks["bf16_tflops_sustained"]
        tc_ms = gemm["total_ms"] + fused["total_ms"]
        tc_flops = gemm["flops"] + fused["flops"]

        def tf(v):
            return v["flops"] / (v["total_ms"] * 1e-3) / 1e12 if v["total_ms"] > 0 else 0.0
        ach = tc_flops / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
        traffic = None          # DRAM bytes per launch of the dominant kernel from the committed ncu capture of this same step
        tpath = os.path.join(ROOT, "profiles", "r2_ncu_gemm_traffic.json")
        if os.path.isfile(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get("dram_bytes_per_launch")
        roofline = {"kernel": "tcgen05 kernels: linear_tc_kernel (bf16 GEMM + fused epilogue; C >= 640 levels) and fused_module_kernel (the whole "
                              "C = 320 module in one kernel)",
                    "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf if peak_tf else None,
                    "frac_of_sustained_peak": ach / peaks["bf16_tflops_sustained"] if peaks.get("bf16_tflops_sustained") else None,
                    "traffic": traffic,
                    "traffic_note": "dram__bytes_read+write per linear_tc_kernel launch, ncu capture of this step (profiles/); "
                                    "algorithmic bytes per launch = %.1f MB" % (gemm["bytes"] / max(gemm["launches"], 1) / 1e6),
                    "peak_source": peaks["source"] + ", bf16_tflops (burst)", "launches": gemm["launches"] + fused["launches"],
                    "per_kernel": {"linear_tc_kernel": {"launches": gemm["launches"], "ms_per_step": gemm["total_ms"] / args.steps, "tflops": tf(gemm),
                                                        "frac": tf(gemm) / peak_tf if peak_tf else None},
                                   "fused_module_kernel": {"launches": fused["launches"], "ms_per_step": fused["total_ms"] / args.steps, "tflops": tf(fused),
                                                           "frac": tf(fused) / peak_tf if peak_tf else None,
                                                           "hbm_GBps": fused["bytes"] / (fused["total_ms"] * 1e-3) / 1e9 if fused["total_ms"] > 0 else None}},
                    "measured_over": f"a second pass of the same {args.steps} steps with a CUDA-event pair around every kernel launch "
                                     f"({ms_profiled / args.steps:.3f} ms/step with the events in the stream)",
                    "share_of_step": tc_ms / ms_profiled if ms_profiled else None,
                    "other_kernels": {k: {"launches": v["launches"], "ms_per_step": v["total_ms"] / args.steps,
                                          "GBps": (v["bytes"] / (v["total_ms"] * 1e-3) / 1e9) if v["total_ms"] > 0 else None,
                                          "frac_of_hbm_peak": (v["bytes"] / (v["total_ms"] * 1e-3) / 1e9 / peaks["hbm_gbs"]) if v["total_ms"] > 0 and peaks["hbm_gbs"] else None}
                                      for k, v in prof.items() if v["launches"] and k not in ("linear_bf16_tcgen05", "fused_module_tcgen05")}}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            flops, run, desc = cpu_reference_time("step", threads)
            secs = run()
            cpu = {"value": flops / secs / 1e12, "unit": UNIT, "cores": threads, "kind": "port", "sample": desc + f" ({secs:.1f} s)"}
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16",
                "data": "synthetic", "config": workload_config(world), "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": d2h_bytes,
                        "copies_alone_ms_per_step": copy_ms, "e2e_over_copies_alone": e2e_ms / copy_ms if copy_ms else None,
                        "runs_ms_per_step": e2e_runs,
                        "note": "PCIe-bound when copies_alone_ms_per_step >= ms_per_step of the device-resident arm: the step's inputs and outputs "
                                "(h2d + d2h bytes) cross the host link inside the timed region, both directions concurrently"},
                "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
                "gpu_eager_baseline": None if eager is None else dict(eager, note="the oracle port's op sequence (= the reference's torch calls) on CUDA tensors under "
                                                                                   "stock torch eager on this GPU, same step; fp32 with TF32 off"),
                "clips": None if args.no_clips else {
                    "metric": "25-step video clips/s, motion modules only", "value": world * 1e3 / clip_ms, "unit": "clips/s", "ms_per_clip": clip_ms,
                    "tflops": world * clip_flops / (clip_ms * 1e-3) / 1e12,
                    "e2e": {"value": world * ce_n / ce_secs if ce_secs else None, "unit": "clips/s", "clips_per_rank": ce_n, "seconds": ce_secs,
                            "h2d_bytes_per_clip": ce_h2d, "d2h_bytes_per_clip": ce_d2h,
                            "what": "per clip: pinned H2D of latents + conditioning, 25 graph-replayed steps (28 motion-module calls + fused CFG/DDIM "
                                    "update), a [3,16,256,256] fp16 frame tensor D2H; ONE NCCL gather of all ranks' frames at the end "
                                    "(sharding.gather_clips); all inside the timed region, max over ranks"},
                    "batch4": {"value": world * 4e3 / clip4_ms, "unit": "clips/s", "ms_per_4_clips": clip4_ms,
                               "tflops": world * clip4_flops / (clip4_ms * 1e-3) / 1e12,
                               "workload": "BASELINE configs[3] shape: the same loop with 4 clips per GPU (CFG batch 8)"},
                    "workload": "BASELINE configs[2] shape: 25 DDIM steps x (20 UNet + 8 SparseCtrl ControlNet motion-module calls), CFG batch 2, "
                                "16 frames, 32x32 latent, bf16; one step captured in a CUDA graph; the rest of the UNet is outside the path"},
                "spatial_transformer": spatial,
                "unet_step_transformers": None if not spatial or "ms_per_step" not in spatial else {
                    "what": "both transformer families of the same UNet step: 20 motion-module calls (`value`) + 16 spatial Transformer3DModel calls",
                    "ms_per_step": ms_step + spatial["ms_per_step"],
                    "tflops": (flops_step + spatial["flops_per_step"]) / ((ms_step + spatial["ms_per_step"]) * 1e-3) / 1e12,
                    "gpu_eager_ms_per_step": (eager["bf16"]["ms_per_step"] + spatial["gpu_eager_baseline"]["ms_per_step"])
                    if eager and "bf16" in eager and "ms_per_step" in spatial.get("gpu_eager_baseline", {}) else None},
                "flops_per_step": flops_step}
        print(json.dumps(line), flush=True)
        if dumped is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for i, (c, a) in enumerate(zip(calls, dumped)):
                np.save(os.path.join(args.dump_outputs, f"call{i:02d}_c{c.channels}_{c.side}x{c.side}.npy"), a)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
