"""Benchmark of the denoising hot path (BASELINE.json metric: denoise-steps/sec, 16 f x 512^2 SD-1.5 UNet3D).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl native|reference] [--dump-outputs DIR] [--profile-dir DIR]

One "step" = one loop body of the reference pipeline (pipelines/pipeline_videoswap.py:556-587): CFG batch
duplication, AnimateDiffUNet3DModel forward on [2,4,16,64,64], CFG combine, DDIM update.  Workload = BASELINE config
"16-frame 512x512 ... 1xB200 fp16" with ED-LoRA per-layer embeddings and adapter residuals active (superset of
configs[1] and configs[2]); synthetic inputs, seeded random weights of the real architecture (no checkpoints offline).
N > 1 (default --mode shard): one process per GPU (torchrun), ONE video split over the ranks -- strong scaling: N = 2 the two
CFG halves (one all-gather of the noise predictions per step), N = 4 / 8 CFG x 2 / 4 frame shards (GroupNorm-statistics
all-reduces + frames<->pixels all-to-all around the motion modules, NCCL over NVLink, captured in the CUDA graph);
`value` = steps of that one video per second.  --mode replicas: one video per rank (weak scaling, no data-path
collective).  Barrier + device timing, max over ranks.

The benchmark writes nothing into the source tree (it may be read-only): --dump-outputs DIR writes the latents the timed
path returned in its last step as DIR/latents.npy (float32; one file per rank, latents_rank<r>.npy, when N > 1), and
--profile-dir DIR the per-shape kernel profile CSV.  Weights and inputs come from fixed seeds, so two builds run with the
same arguments can be compared output for output.  The GroupNorm statistics are summed with float atomics, so two runs of
one build already differ in the last bits: 76 dB PSNR between the dumps of two `--steps 10 --warmup 3` runs (B200, 1000 W
power limit).
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "denoise-steps/sec, 16f 512^2 SD1.5 UNet3D (CFG UNet fwd + CFG combine + DDIM step)"
UNIT = "steps/s"
FLOP_PER_STEP = 35.26e12          # algorithmic FLOPs of one CFG step at this config (SURVEY.md 8d)
FRAMES, LATENT = 16, 64
CATS = ["gemm", "conv3x3", "attention", "temporal_attention", "groupnorm", "layernorm", "other"]
DUMP_LIMIT = 64 << 20             # bytes of --dump-outputs per run


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """Writes each tensor as <out_dir>/<name>.npy in float32.  When they exceed `limit` bytes in all, each is replaced by
    the same fixed, seeded sample of its flattened elements (sorted positions), so that runs stay comparable."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: v.detach().float().cpu().numpy() for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        if total > limit:
            keep = a.size * limit // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return {"tflops": d.get("bf16_tflops_sustained", d.get("bf16_tflops", 1590.0)), "tflops_burst": d.get("bf16_tflops", 1590.0),
                "gbs": d.get("hbm_gbs", 6650.0), "source": "MEASURED_PEAKS.json (sustained bf16 cuBLAS / copy)"}
    return {"tflops": 1400.0, "tflops_burst": 1590.0, "gbs": 6650.0, "source": "fallback (B200_PROFILING.md)"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i] == "Active" for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def gpu_weights(cfg, device):
    """Random weights of the real architecture generated directly on the GPU (values are irrelevant for timing)."""
    import torch
    from videoswap_b200 import unet_param_shapes
    from videoswap_b200.weights import temporal_pe_table
    g = torch.Generator(device=device).manual_seed(0)
    sd = {}
    for name, shape in unet_param_shapes(cfg).items():
        if name.endswith(".pe"):
            sd[name] = temporal_pe_table(shape[1], shape[2]).to(device)
        elif len(shape) >= 2:
            fan_in = math.prod(shape[1:])
            sd[name] = ((torch.rand(shape, device=device, generator=g) * 2 - 1) / math.sqrt(fan_in)).half()
        elif name.endswith(".weight"):
            sd[name] = (1 + 0.1 * torch.randn(shape, device=device, generator=g)).half()
        else:
            sd[name] = (0.02 * torch.randn(shape, device=device, generator=g)).half()
    return sd


def cpu_oracle_sample(frames=2, latent=LATENT, reps_budget_s=15.0, warmup=1, max_reps=5):
    """Times the CPU oracle (restatement of the reference's UNet forward) on a bounded sample of the workload:
    one UNet forward on [1,4,frames,latent,latent] with ED-LoRA embeddings = frames/16 of one half of a CFG step."""
    import torch
    from oracle import unet3d_oracle as O
    from videoswap_b200 import UNetConfig, seeded_state_dict, unet_param_shapes
    # measured on the 128-core GPU box (tools/cpu_thread_sweep.py): 16 threads 5.8 s, 32: 6.0 s, 64: 8.9 s, 128: 138 s per
    # sample -- the sample's tensors are too small for more threads, so the baseline uses the fastest setting
    torch.set_num_threads(min(os.cpu_count() or 1, 16))
    sd = seeded_state_dict(unet_param_shapes(UNetConfig()), seed=0)
    x = torch.randn(1, 4, frames, latent, latent)
    ehs = torch.randn(1, 16, 77, 768)
    times = []
    with torch.no_grad():
        for _ in range(warmup):
            O.unet_forward(sd, O.OracleConfig(), x, 981, ehs)
        t_total = 0.0
        while len(times) < max_reps and (t_total < reps_budget_s or not times):
            t0 = time.perf_counter()
            O.unet_forward(sd, O.OracleConfig(), x, 981, ehs)
            times.append(time.perf_counter() - t0)
            t_total += times[-1]
    frac = frames / (2.0 * FRAMES)                 # fraction of one CFG step (B=2 x 16 frames) this sample covers
    return times, frac


def library_baseline(sd16, dev, lat0, embeds, residuals, ts, native_out, steps=5, warmup=2):
    """The bar BASELINE.md section 3 names: the SAME step (the oracle's functional restatement of the reference graph) in
    fp16 through stock PyTorch eager on this GPU -- cuDNN convolutions, cuBLASLt linears, F.scaled_dot_product_attention,
    aten GroupNorm/LayerNorm -- timed with CUDA events outside the native timed regions.  Reported only.  Also returns the
    PSNR between the two fp16 implementations' step outputs at the full benchmark size."""
    import math
    import torch
    from oracle import unet3d_oracle as O
    O.USE_SDPA = True
    sched = O.DDIM()
    cfgo = O.OracleConfig()
    sd = {k: (v if v.dtype == torch.float16 else v.half()) for k, v in sd16.items() if not k.endswith(".pe")}
    res = [r for r in residuals]

    def step(lat, t):
        eps2 = O.unet_forward(sd, cfgo, torch.cat([lat] * 2), t, embeds, res)
        return sched.step(O.cfg_combine(eps2.float(), 7.5), t, lat.float(), 50).half()

    try:
        with torch.no_grad():
            lat = lat0
            for i in range(warmup):
                out = step(lat, ts[i % len(ts)])
            torch.cuda.synchronize()
            first = step(lat0, ts[0])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(steps):
                lat = step(lat, ts[(warmup + i) % len(ts)])
            e1.record()
            torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        d = (native_out.float() - first.float())
        rng = float(first.float().max() - first.float().min())
        mse = float((d ** 2).mean())
        return {"value": 1e3 / ms, "unit": UNIT, "ms_per_step": ms, "steps": steps, "dtype": "f16",
                "how": "oracle graph (restatement of the reference modules) on cuda fp16, torch eager: cuDNN conv2d, cuBLASLt "
                       "linear, F.scaled_dot_product_attention, aten group_norm/layer_norm; same weights/inputs as the native arm",
                "torch": torch.__version__, "native_vs_library_step_psnr_db": 10 * math.log10(rng * rng / mse) if mse > 0 else float("inf")}
    except Exception as e:  # noqa: BLE001  (reported-only arm: never take the native numbers down with it)
        return {"unavailable": repr(e)[:300]}
    finally:
        O.USE_SDPA = False


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path.  The reference is pure Python on diffusers (not installable offline)
    and /root/reference does not travel to the GPU box, so this times oracle/ (the pinned CPU restatement) on the host
    cores; rank 0 only."""
    if rank != 0:
        return
    import torch
    # bounded: at most `steps` samples and ~90 s of CPU time in total, so the arm always ends within a few minutes
    times, frac = cpu_oracle_sample(frames=2, reps_budget_s=90.0, warmup=min(args.warmup, 1), max_reps=max(args.steps, 1))
    t = sorted(times)[len(times) // 2]
    v = frac / t
    sample = "oracle UNet forward fp32 on [1,4,2,64,64] + ED-LoRA embeds = 1/16 of a CFG step; value = (1/16)/median time"
    print(json.dumps({
        "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times), "warmup": min(args.warmup, 1),
        "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "impl": "reference",
        "config": {"workload": "16f 512^2 CFG denoise step (configs[1]/[2]); CPU arm runs a 2-frame no-CFG sample"},
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time eager launches instead of the CUDA-graph replay")
    ap.add_argument("--no-library-baseline", action="store_true", help="skip the torch-eager fp16 arm (reported-only)")
    ap.add_argument("--no-inversion", action="store_true", help="skip the B=1 DDIM-inversion extra (reported-only)")
    ap.add_argument("--frames", type=int, default=FRAMES)
    ap.add_argument("--latent-h", type=int, default=LATENT, help="latent height (extra configs, e.g. 56 for 448x768 video)")
    ap.add_argument("--latent-w", type=int, default=LATENT, help="latent width (e.g. 96)")
    ap.add_argument("--mode", default="shard", choices=["shard", "replicas"],
                    help="multi-GPU scheme: ONE video split over the ranks (CFG halves x frame shards; strong scaling, "
                         "default) or independent videos per rank (weak scaling)")
    ap.add_argument("--option", action="append", default=[], help="kernel A/B switch name=value (vs_set_option)")
    ap.add_argument("--tag", default="", help="suffix of the per-shape profile CSV")
    ap.add_argument("--profile-dir", help="write the per-shape profile CSV (profile_shapes_n<N><tag>.csv) of the eager pass here")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the latents of the last timed step as DIR/latents.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl native (the reference arm times a CPU sample, not the step)")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from videoswap_b200 import AnimateDiffUNet3DModel, DDIMScheduler, VideoSwapPipeline, _lib, dist_util, ops
    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    W = max(args.warmup, 3)
    K = args.steps
    sharded = args.mode == "shard" and world > 1
    cfg_split = sharded                             # (name kept for the JSON fields below)
    plan = dist_util.make_plan(world, rank, cfg=True) if sharded else dist_util.ShardPlan()
    seed_rank = 0 if sharded else rank              # all ranks work on the SAME video
    Fr = args.frames

    model = AnimateDiffUNet3DModel(init="empty")
    sd16 = gpu_weights(model.cfg, dev)
    model.load_state_dict(sd16, assign=True)
    pipe = VideoSwapPipeline(model, DDIMScheduler())
    pipe.scheduler.set_timesteps(50)
    ts = pipe.scheduler.timesteps
    g = torch.Generator(device=dev).manual_seed(100 + seed_rank)
    LH, LW = args.latent_h, args.latent_w
    lat0 = torch.randn((1, 4, Fr, LH, LW), device=dev, generator=g).half()
    embeds = torch.randn((2, 16, 77, 768), device=dev, generator=g).half()
    boc = model.cfg.block_out_channels
    residuals = [(0.1 * torch.randn((2 * Fr, c, LH >> l, LW >> l), device=dev, generator=g)).half() for l, c in enumerate(boc)]
    res_loc = None
    if sharded:
        plan = dist_util.create_comms(plan)
        dist_util.attach(model, plan)
        lat0 = plan.shard_frames(lat0, 2)                                       # this rank's frames of the one video
        res_loc = [plan.shard_frame_major(r[:Fr], Fr) for r in residuals]       # per-frame maps (identical for both CFG halves)

    def step(lat, i):
        if sharded:
            return pipe.step_sharded(lat, ts[i % len(ts)], embeds, 7.5, plan, res_loc)
        return pipe.step(lat, ts[i % len(ts)], embeds, 7.5, list(residuals))

    lib = _lib.lib()
    for opt in args.option:
        name, val = opt.split("=")
        _lib.call("vs_set_option", name.encode(), int(val))
    lat = lat0
    for i in range(W):
        lat = step(lat, i)
    torch.cuda.synchronize()

    # ---------------- timed region 1: inputs resident in HBM, per-launch CUDA-event profile for the roofline numbers
    lib.vs_profile_reset()
    lib.vs_profile_enable(1)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = lib.vs_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    torch.cuda.nvtx.range_push("vs_timed_eager")      # lets `ncu --nvtx --nvtx-include vs_timed_eager/` pick this region
    for i in range(K):
        lat = step(lat, W + i)
    torch.cuda.nvtx.range_pop()
    e1.record()
    torch.cuda.synchronize()
    launches = lib.vs_launch_count() - n0
    lib.vs_profile_enable(0)
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.barrier()
        ms = t.item()
    prof = {}
    for ci, name in enumerate(CATS):
        a, b, c = C.c_double(), C.c_double(), C.c_longlong()
        _lib.call("vs_profile_collect", ci, C.byref(a), C.byref(b), C.byref(c))
        prof[name] = {"ms_per_step": a.value / K, "work_per_step": b.value / K, "launches_per_step": c.value / K}
    if rank == 0 and args.profile_dir:
        os.makedirs(args.profile_dir, exist_ok=True)
        _lib.call("vs_profile_dump", os.path.join(args.profile_dir, f"profile_shapes_n{world}{args.tag}.csv").encode())
    lib.vs_profile_reset()
    finite = bool(torch.isfinite(lat).all().item())
    ms_eager = ms
    last_out = lat.clone() if args.dump_outputs else None    # the timed path's result when there is no graph

    # ---------------- timed region 1b (the reported `value`): the same step captured in a CUDA graph and replayed
    gstep = None
    if not args.no_graph:
        from videoswap_b200.pipeline import GraphedStep
        gstep = GraphedStep(pipe, lat0, embeds, 7.5, res_loc if sharded else residuals, plan=plan if sharded else None)
        lat = lat0
        for i in range(W):
            lat = gstep(lat, ts[i % len(ts)])
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for i in range(K):
            lat = gstep(lat, ts[(W + i) % len(ts)])
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if args.dump_outputs:
            last_out = lat.clone()           # the graph's output buffer is overwritten by the end-to-end pass below
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = t.item()
        finite = finite and bool(torch.isfinite(lat).all().item())

    clocks = sampler.stop() if rank == 0 else None     # sampled across both device-timed regions (eager profile + graph)
    # ---------------- timed region 2: end to end through the public API with HOST buffers (pinned), H2D + D2H inside
    h_lat = lat0.cpu().pin_memory()
    h_emb = embeds.cpu().pin_memory()
    h_out = torch.empty_like(h_lat).pin_memory()
    d_lat = torch.empty_like(lat0)
    d_emb = gstep.embeds if gstep is not None else torch.empty_like(embeds)

    def e2e_step(i):
        d_lat.copy_(h_lat, non_blocking=True)
        d_emb.copy_(h_emb, non_blocking=True)
        if gstep is not None:
            out = gstep(d_lat, ts[i % len(ts)])
        else:
            out = step(d_lat, i)
        h_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()      # the caller reads the result on the host every step
        h_lat.copy_(h_out)

    for i in range(2):
        e2e_step(i)
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    e0.record()
    for i in range(K):
        e2e_step(i)
    e1.record()
    torch.cuda.synchronize()
    ms_e2e = max(e0.elapsed_time(e1), (time.perf_counter() - t0) * 1e3)
    if world > 1:
        t = torch.tensor([ms_e2e], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_e2e = t.item()

    # ---------------- extra (reported only): the DDIM-inversion step (SURVEY 8f-1): B = 1, no CFG, 17.67 TFLOP -- half of
    # the UNet calls of one `test.py` edit.  Its own CUDA graph; the CFG graph above stays valid (shared, pinned arena).
    inversion = None
    if not args.no_inversion and gstep is not None and not cfg_split and (LH, LW) == (LATENT, LATENT):
        from videoswap_b200.pipeline import GraphedStep
        inv = GraphedStep(pipe, lat0, embeds[1:2, 0].contiguous(), 1.0, None, inverse=True)
        its = pipe.inverse_scheduler.timesteps
        lat = lat0
        for i in range(W):
            lat = inv(lat, its[i % len(its)])
        torch.cuda.synchronize()
        e0.record()
        for i in range(K):
            lat = inv(lat, its[(W + i) % len(its)])
        e1.record()
        torch.cuda.synchronize()
        ms_inv = e0.elapsed_time(e1) / K
        inversion = {"ms_per_step": ms_inv, "steps_per_s": 1e3 / ms_inv, "tflops": round(17.674e12 * (Fr / FRAMES) / (ms_inv / 1e3) / 1e12, 1),
                     "config": f"latents [1,4,{Fr},{LH},{LW}], no CFG (UNet batch 1), prompt embeds [1,77,768], inverse DDIM step, CUDA graph",
                     "finite": bool(torch.isfinite(lat).all().item())}
        del inv

    library = None
    if rank == 0 and world == 1 and not args.no_library_baseline and gstep is not None:
        native_first = gstep(lat0, ts[0]).clone()
        library = library_baseline(sd16, dev, lat0, embeds, residuals, ts, native_first, steps=min(K, 5))

    if rank == 0:
        pk = peaks()
        jobs = 1 if cfg_split else world            # videos denoised concurrently
        value = jobs * K / (ms / 1e3)
        e2e = jobs * K / (ms_e2e / 1e3)
        tensor_cats = ["gemm", "conv3x3", "attention"]
        # dominant kernel: gemm_tc_kernel -- one template serves the GEMMs and the implicit-GEMM 3x3 convs, so its launches
        # of both categories are pooled: achieved = algorithmic FLOPs per launch / average launch duration
        g_ms = prof["gemm"]["ms_per_step"] + prof["conv3x3"]["ms_per_step"]
        g_work = prof["gemm"]["work_per_step"] + prof["conv3x3"]["work_per_step"]
        g_n = prof["gemm"]["launches_per_step"] + prof["conv3x3"]["launches_per_step"]
        if g_ms >= prof["attention"]["ms_per_step"]:
            dom_name, d = "gemm_tc_kernel (GEMM + implicit-GEMM 3x3 conv)", {"ms_per_step": g_ms, "work_per_step": g_work, "launches_per_step": g_n}
        else:
            dom_name, d = "attn_tc_kernel", prof["attention"]
        ach = d["work_per_step"] / (d["ms_per_step"] / 1e3) / 1e12 if d["ms_per_step"] > 0 else 0.0
        traffic, traffic_src = None, None
        summ = os.path.join(ROOT, "profiles", "r02_launches_summary.json")
        if not os.path.exists(summ):
            summ = os.path.join(ROOT, "profiles", "r01_launches_summary.json")
        if os.path.exists(summ):      # DRAM bytes per launch of the same kernel from the committed ncu capture of one step
            with open(summ) as f:
                ks = json.load(f)["kernels"]
            sel = [v for k, v in ks.items() if k.startswith(dom_name.split(" ")[0])]
            if sel:
                traffic = sum((v["dram_read_MB"] + v["dram_write_MB"]) * 1e6 for v in sel) / sum(v["launches"] for v in sel)
                traffic_src = f"profiles/{os.path.basename(summ)} (ncu dram__bytes_read.sum + dram__bytes_write.sum, cold L2)"
        kernels = {}
        for n, p_ in prof.items():
            if p_["ms_per_step"] <= 0:
                continue
            rate = p_["work_per_step"] / (p_["ms_per_step"] / 1e3)
            if n in tensor_cats:
                kernels[n] = {"ms_per_step": round(p_["ms_per_step"], 3), "tflops": round(rate / 1e12, 1),
                              "frac_of_peak": round(rate / 1e12 / pk["tflops"], 3), "launches": p_["launches_per_step"]}
            else:
                kernels[n] = {"ms_per_step": round(p_["ms_per_step"], 3), "gbs": round(rate / 1e9, 1),
                              "frac_of_peak": round(rate / 1e9 / pk["gbs"], 3), "launches": p_["launches_per_step"]}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
            "ms_per_step": ms / K, "higher_is_better": True, "scaling": "strong" if cfg_split else "weak", "vs_baseline": None, "dtype": "f16",
            "data": "synthetic",
            "config": {"workload": f"{Fr}-frame {8 * LH}x{8 * LW} (latent [1,4,{Fr},{LH},{LW}]), CFG 7.5 (UNet batch 2), ED-LoRA embeds "
                                   f"[2,16,77,768], adapter residuals active, DDIM step; " +
                                   (f"ONE video over {world} GPUs: CFG halves x {plan.frame_shards} frame shard(s); exchanges per step: 1 all-gather of eps"
                                    + (", 45 GroupNorm-statistics all-reduces, 40 frames<->pixels all-to-alls (NCCL, inside the CUDA graph)" if plan.frame_shards > 1 else "")
                                    if sharded else "one video per GPU"),
                       "parallelism": (f"cfg2 x frames{plan.frame_shards}" if sharded else f"replicas x{world}"),
                       "timing": "CUDA events; working set (2.55 GB weights + activations) >> 126 MB L2, no flush needed; "
                                 "`value`/`e2e` replay the step as a CUDA graph, the per-kernel profile comes from an eager pass "
                                 "of the same K steps with per-launch events",
                       "eager_ms_per_step": round(ms_eager / K, 3), "cuda_graph": gstep is not None,
                       "whole_step_tflops": (round(FLOP_PER_STEP * (Fr / FRAMES) * value / 1e12, 1)
                                             if (LH, LW) == (LATENT, LATENT) else None)},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": (h_lat.numel() * 2 + h_emb.numel() * 2) * world,
                    "d2h_bytes_per_step": h_out.numel() * 2 * world},     # every rank moves its own latents (shard) + embeddings
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"kernel": dom_name, "bound": "tensor", "achieved": ach, "peak": pk["tflops"], "unit": "TFLOP/s",
                         "frac": ach / pk["tflops"], "traffic": traffic, "traffic_source": traffic_src,
                         "launches_per_step": d["launches_per_step"],
                         "flops_per_launch": d["work_per_step"] / max(d["launches_per_step"], 1),
                         "avg_launch_us": 1e3 * d["ms_per_step"] / max(d["launches_per_step"], 1), "peak_source": pk["source"]},
            "kernels": kernels, "finite": finite,
            "library_baseline": library, "inversion_step": inversion,
        }
        if library and "value" in library:
            out["vs_library"] = {"device_ratio": value / library["value"], "e2e_ratio": e2e / library["value"]}
        if world == 1 and not args.no_cpu_baseline:
            times, frac = cpu_oracle_sample(frames=2, reps_budget_s=12.0)
            tmed = sorted(times)[len(times) // 2]
            out["cpu_baseline"] = {"value": frac / tmed, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                   "sample": f"oracle UNet fwd fp32 on [1,4,2,64,64] (1/16 CFG step), median of {len(times)} reps = {tmed:.2f} s"}
        else:
            out["cpu_baseline"] = None
        print(json.dumps(out))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latents" if world == 1 else f"latents_rank{rank}": last_out}, DUMP_LIMIT // world)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    sys.dont_write_bytecode = True    # the package is imported inside main(): no __pycache__ in the tree the benchmark runs from
    main()
