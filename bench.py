#!/usr/bin/env python
"""bench.py — frames/s of the TokenFlow edit on B200(s).  Default workload = BASELINE.json configs[1] ("C2"):
40-frame 512x512 SD1.5 PnP 50-step edit, keyframe stride B=8 -> K=5 keyframes per step, random-init
SD1.5-shape UNet in fp16, synthetic latents (no SD weights / VAE / CLIP exist offline).

A "step" is one denoising step of the edit = the pivotal samples (extended attention, caches filled) + all
frames (NN field + propagation) + CFG + DDIM update.  frames/s = N / (n_steps * mean step time), measured over
--steps consecutive denoising steps.

  python bench.py [--gpus N --steps K --warmup W]            our arm (CUDA kernels, sm_100a), config C2
  python bench.py --config {C2,C3,C4,C5s4,C5s8,C5s16}        the other BASELINE.json configs
  python bench.py --verify                                   + N-rank vs 1-rank (and graph vs eager) result check
  python bench.py --impl reference ...                       the reference's algorithm on host cores
  python bench.py --dump-outputs DIR                         + DIR/latents.npy: what the last timed step returned

One JSON line on stdout (rank 0).  Keys follow the driver contract; `roofline` describes the dominant hot-path
kernel (per-launch CUDA events inside the timed region: event-record nodes of the captured step graphs, max over
ranks), `cpu_baseline` the oracle port timed on the host cores on a bounded sample, `e2e` the same metric through
the public editor call with pinned HOST latents (H2D + D2H inside the timed region), `gpu_reference` the
reference's own GPU arithmetic (oracle ops on CUDA under autocast, eager, the reference's pass schedule).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)

# BASELINE.json configs (SURVEY.md §8d).  n_steps = denoising steps of the full edit (SDEdit start=0.9: 44 of 50).
CONFIGS = {
    "C2": dict(kind="sd15", n_frames=40, batch=8, latent=64, mode="pnp", n_timesteps=50, n_steps=50,
               label="C2: 40-frame 512x512 SD1.5 PnP 50-step edit, B=8 (K=5 keyframes)"),
    "C3": dict(kind="sd15", n_frames=80, batch=8, latent=64, mode="pnp", n_timesteps=50, n_steps=50,
               label="C3: 80-frame 512x512 SD1.5 PnP 50-step edit, B=8 (K=10 keyframes)"),
    "C4": dict(kind="sd21", n_frames=40, batch=8, latent=96, mode="sdedit", n_timesteps=50, n_steps=44,
               label="C4: 40-frame 768x768 SD2.1 SDEdit (start 0.9: 44 of 50 steps), B=8 (K=5 keyframes), extended attention "
                     "without PnP injection"),
    "C5s4": dict(kind="sd15", n_frames=200, batch=4, latent=64, mode="pnp", n_timesteps=50, n_steps=50,
                 label="C5: 200-frame 512x512 SD1.5 PnP edit, keyframe stride 4 (K=50 keyframes)"),
    "C5s8": dict(kind="sd15", n_frames=200, batch=8, latent=64, mode="pnp", n_timesteps=50, n_steps=50,
                 label="C5: 200-frame 512x512 SD1.5 PnP edit, keyframe stride 8 (K=25 keyframes)"),
    "C5s16": dict(kind="sd15", n_frames=192, batch=16, latent=64, mode="pnp", n_timesteps=50, n_steps=50,
                  label="C5: 192-frame (200 truncated to a multiple of 16) 512x512 SD1.5 PnP edit, keyframe stride 16 (K=12)"),
}
METRIC_C2 = "frames/sec for 40-frame 512x512 SD1.5 50-step edit"
TENSOR_KERNELS = ("tf_ext_attn", "tf_nn_field")


def metric_name(cfg_name):
    c = CONFIGS[cfg_name]
    if cfg_name == "C2":
        return METRIC_C2
    px = c["latent"] * 8
    return f"frames/sec for {c['n_frames']}-frame {px}x{px} {'SD1.5' if c['kind'] == 'sd15' else 'SD2.1'} {c['n_steps']}-step edit"


def workload(cfg_name):
    return CONFIGS[cfg_name]["label"] + ", random-init UNet fp16, synthetic latents"


# ------------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------------
def measured_peaks():
    path = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"hbm_gbs": p["hbm_gbs"], "tf_burst": p["bf16_tflops"], "tf_sustained": p.get("bf16_tflops_sustained", p["bf16_tflops"]),
                "source": "measured"}
    return {"hbm_gbs": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi clocks + throttle reasons every 200 ms while the timed region runs."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.gpu_index)], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); smax.append(float(parts[2])); power.append(float(parts[3]))
            except ValueError:
                continue
            for name, val in zip(names, parts[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def dump_outputs(out_dir, arrays, limit=64 << 20):
    """Write each array as <out_dir>/<name>.npy in float32, for comparing two builds output for output."""
    import numpy as np
    host = {name: t.detach().float().cpu().numpy() for name, t in arrays.items()}
    total = sum(a.nbytes for a in host.values())
    assert total <= limit, f"outputs are {total} bytes, more than {limit}"
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def dist_env():
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def build_editor(device, cfg_name="C2", world=1, rank=0, seed=1, channels_last=True, frames_per_pass=None, fused_pass=True,
                 cuda_graph=True, hooks=None, unet=None, check_keyframes=False, comm=None, dual_stream=None):
    from tokenflow_b200 import sd_unet, tokenflow_utils as tfu
    from tokenflow_b200.editor import TokenFlowEditor, synthetic_inputs
    from tokenflow_b200.scheduler import DDIMScheduler
    c = CONFIGS[cfg_name]
    if unet is None:
        # multi-GPU: draw the weights on the device (torchrun pins OMP_NUM_THREADS=1 and a CPU init of the 860M
        # parameters then takes minutes per rank); single GPU keeps the device-independent CPU init
        unet = sd_unet.build_unet(c["kind"], seed=seed, device=device, dtype=torch.float16, init_on_device=world > 1)
        if channels_last:
            unet = unet.to(memory_format=torch.channels_last)
    cfg = {"n_frames": c["n_frames"], "batch_size": c["batch"], "n_timesteps": c["n_timesteps"], "guidance_scale": 7.5,
           "mode": c["mode"], "pnp_attn_t": 0.5, "pnp_f_t": 0.8, "start": 0.9,
           "frames_per_pass": frames_per_pass if frames_per_pass else c["n_frames"],
           "fused_pass": bool(fused_pass), "cuda_graph": bool(cuda_graph), "keyframe_seed": seed,
           "check_keyframes": bool(check_keyframes), "dual_stream": dual_stream}
    x, text, pnp, src = synthetic_inputs(c["n_frames"], c["latent"], unet.config.cross_attention_dim, c["n_timesteps"],
                                         seed=seed, device=device, dtype=torch.float16)
    ed = TokenFlowEditor(unet, DDIMScheduler(), hooks or tfu, cfg, text, pnp, source_latents=lambda t: src[t],
                         world_size=world, rank=rank)
    if comm is not None:
        ed.attach_communicator(comm)
    ed.init_method()
    return ed, x, src


def collect_nn_indices(ed):
    """Per TokenFlow block, the int32 NN indices the last step produced for this rank's frames."""
    out = []
    for blk in ed.hooks._transformer_blocks(ed):
        idx = getattr(blk, "_tf_nn_idx", None)
        if idx is not None:
            out.append(tuple(None if t is None else t.detach().clone() for t in idx))
    return out


def run_verify(args, device, world, rank, ed, x0, cfg_name, steps=2):
    """Result check before timing: `steps` denoising steps through the measured path (N ranks, CUDA graphs) against
    the same steps run by ONE rank eagerly (every rank runs that single-process reference locally, no
    collectives), same seed and keyframes.  Reports max |difference| of the latents and the NN-index mismatches
    of this rank's frames, reduced over ranks."""
    import torch.distributed as dist
    c = CONFIGS[cfg_name]
    N = c["n_frames"]
    per = N // world
    x = x0.clone()
    for i in range(steps):
        x = ed.step_index(x, i)
    idx_n = collect_nn_indices(ed)
    kf_n = [list(k) for k in ed.keyframe_log[-steps:]]
    ref, xr, _ = build_editor(device, cfg_name, 1, 0, cuda_graph=False, unet=ed.unet)
    for i in range(steps):
        xr = ref.step_index(xr, i)
    idx_1 = collect_nn_indices(ref)
    kf_1 = [list(k) for k in ref.keyframe_log[-steps:]]
    ed.init_method()                                   # the reference editor re-registered hooks on the shared UNet
    diff = (x.float() - xr.float()).abs().max()
    mism = torch.zeros(2, device=device, dtype=torch.float64)
    lo = rank * per
    # frames of the first keyframe batch have no second keyframe: their idx_b rows are never written or read
    has_b = torch.tensor([b >= 0 for b in ed.frame_table(list(range(lo, lo + per)))[1]], device=device)
    for (a_n, b_n), (a_1, b_1) in zip(idx_n, idx_1):
        mism[0] += (a_n != a_1[lo:lo + per]).sum()
        mism[1] += a_n.numel()
        if b_n is not None and b_1 is not None:
            mism[0] += (b_n != b_1[lo:lo + per])[has_b].sum()
            mism[1] += b_n[has_b].numel()
    stats = torch.stack([diff.double(), xr.float().abs().max().double()])
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(mism, op=dist.ReduceOp.SUM)
    # graphs vs eager on the SAME world size (must be identical: same kernels, same order)
    eager, xe, _ = build_editor(device, cfg_name, world, rank, cuda_graph=False, unet=ed.unet, comm=ed.comm,
                                dual_stream=ed.config.get("dual_stream"))
    for i in range(steps):
        xe = eager.step_index(xe, i)
    ed.init_method()
    g_diff = (x.float() - xe.float()).abs().max().double().reshape(1)
    if world > 1:
        dist.all_reduce(g_diff, op=dist.ReduceOp.MAX)
    return {"steps": steps, "world": world, "against": "1 rank, eager, same seed and keyframes (run locally by every rank)",
            "max_abs_diff": float(stats[0]), "ref_absmax": float(stats[1]), "keyframes_equal": kf_n == kf_1,
            "nn_idx_mismatch": int(mism[0]), "nn_idx_total": int(mism[1]),
            "nn_idx_mismatch_frac": float(mism[0] / max(1.0, float(mism[1]))),
            "graph_vs_eager_max_abs_diff": float(g_diff[0])}


def time_gpu_reference(args, device, cfg_name, unet, steps):
    """The reference's GPU arithmetic on the same B200: this repo's hook plumbing with the ORACLE ops (plain
    torch bmm / softmax / argmax / gather, as tokenflow_utils.py:114-199, :329-397 issue them) under
    torch.autocast(fp16), eager, the reference's schedule (pivotal pass + N/B frame passes)."""
    from oracle.oracle_ops import OracleOps
    from tokenflow_b200 import tokenflow_utils as tfu
    c = CONFIGS[cfg_name]
    tfu._install_ops_for_testing(OracleOps())
    try:
        ed, x, _ = build_editor(device, cfg_name, 1, 0, frames_per_pass=c["batch"], fused_pass=False, cuda_graph=False, unet=unet)
        ed.step_index(x, 0)                                     # warm-up
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            x = ed.step_index(x, 1 + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        peak_gb = torch.cuda.max_memory_allocated() / 2 ** 30
    finally:
        tfu._install_ops_for_testing(None)
    return {"what": "reference GPU arithmetic (oracle ops on CUDA, autocast fp16, eager, pivotal pass + N/B frame passes) "
                    "on the same UNet and B200", "steps": steps, "ms_per_step": round(ms, 2),
            "value": round(c["n_frames"] / (c["n_steps"] * ms / 1e3), 4), "unit": "frames/s",
            "peak_mem_gib": round(peak_gb, 1)}


def run_ours(args):
    rank, local_rank, world = dist_env()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    cfg_name = args.config
    c = CONFIGS[cfg_name]
    N, n_steps = c["n_frames"], c["n_steps"]
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    comm = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=device)      # NCCL logs go to stderr; stdout stays the one JSON line
        if not args.torch_collectives:
            from tokenflow_b200.ops import Communicator
            comm = Communicator(world, rank)                    # tf_comm_init / tf_allgather (C ABI)
    from tokenflow_b200 import tokenflow_utils as tfu
    ops = tfu._ops()                                     # CudaOps: raises if the .so / B200 is missing
    torch.backends.cudnn.benchmark = bool(args.cudnn_benchmark)
    ed, x0, src = build_editor(device, cfg_name, world, rank, channels_last=not args.no_channels_last,
                               frames_per_pass=args.frames_per_pass, fused_pass=bool(args.fused_pass),
                               cuda_graph=bool(args.graph), comm=comm,
                               dual_stream=None if args.dual_stream < 0 else bool(args.dual_stream))
    timesteps = list(ed._t_host)
    n_sched = len(timesteps)

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    ops.enable_timing(not args.no_kernel_events)         # before the first step: graphs capture their event nodes
    verify = None
    if args.verify:
        verify = run_verify(args, device, world, rank, ed, x0, cfg_name)
        ops.timing_summary()                             # drop the events of the verify run's eager steps

    # ---- device-resident measurement (`value`) ----
    x = x0.clone()
    for i in range(args.warmup):
        x = ed.step_index(x, i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = ops.launch_count()
    if args.graph:
        ed.mark_graph_replays()                          # kernel times below cover the timed replays only
    else:
        ops.timing_summary()                             # drop the warm-up's events
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps):
        x = ed.step_index(x, args.warmup + i)
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = ops.launch_count() - launches0
    if args.graph:
        # launches replayed from the graphs are not counted by the library's counter: count the graphs' kernel nodes
        kernel_times, graph_steps = ed.graph_kernel_times(since_mark=True)     # replays of the timed region
        launches = sum(k_["launches"] for k_ in kernel_times.values()) if kernel_times else \
            ed.graph_launches_per_step() * args.steps
        per_step_div = float(max(1, graph_steps)) if kernel_times else float(args.steps)
    else:
        kernel_times = ops.timing_summary()
        per_step_div = float(args.steps)
    ops.enable_timing(False)
    clocks = sampler.stop() if rank == 0 else None
    finite = bool(torch.isfinite(x.float()).all().item())
    if args.dump_outputs and rank == 0:
        # the denoised latents of every frame (all-gathered when sharded), as the step returns them to its caller
        dump_outputs(args.dump_outputs, {"latents": x})

    # ---- end-to-end through the public call with pinned host latents (`e2e`) ----
    ms_e2e = float("nan")
    if not args.skip_e2e:
        x_host = x0.cpu().pin_memory()
        src_host = {t: v.cpu().pin_memory() for t, v in src.items()}
        out_host = torch.empty_like(x_host).pin_memory()
        for i in range(min(args.warmup, 3)):
            ed.edit_step_host(x_host, src_host[timesteps[i % n_sched]], timesteps[i % n_sched], out_host)
            x_host.copy_(out_host)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(args.steps):
            t = timesteps[(args.warmup + i) % n_sched]
            ed.edit_step_host(x_host, src_host[t], t, out_host)
            x_host.copy_(out_host)
        e1.record()
        barrier()
        ms_e2e = e0.elapsed_time(e1)

    # ---- max over ranks: step time and every hot-path kernel's time ----
    names = sorted(kernel_times.keys())
    kt_rank0 = {k_: dict(v_) for k_, v_ in kernel_times.items()}
    if world > 1:
        import torch.distributed as dist
        tt = torch.tensor([ms_total, ms_e2e], device=device, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_total, ms_e2e = tt.tolist()
        all_names = [None] * world
        dist.all_gather_object(all_names, names)
        names = sorted(set().union(*all_names))
        vals = torch.tensor([[kernel_times.get(n_, {}).get("ms", 0.0), kernel_times.get(n_, {}).get("work", 0.0),
                              kernel_times.get(n_, {}).get("launches", 0)] for n_ in names], device=device, dtype=torch.float64)
        vmax, vmin = vals.clone(), vals.clone()
        dist.all_reduce(vmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(vmin, op=dist.ReduceOp.MIN)
        # the slowest rank per kernel (its time, with that kernel's max work/launches: an upper bound on time per work)
        kernel_times = {n_: {"ms": float(vmax[j, 0]), "ms_min_rank": float(vmin[j, 0]), "work": float(vmax[j, 1]),
                             "launches": int(vmax[j, 2])} for j, n_ in enumerate(names)}
    gpu_ref = None
    if rank == 0 and world == 1 and args.gpu_reference_steps > 0 and not args.no_gpu_reference:
        try:
            gpu_ref = time_gpu_reference(args, device, cfg_name, ed.unet, args.gpu_reference_steps)
        except Exception as ex:  # noqa: BLE001  (e.g. out of memory at the long-video configs: the reference materialises K copies of K/V)
            gpu_ref = {"unavailable": f"{type(ex).__name__}: {str(ex)[:160]}"}
            torch.cuda.empty_cache()
    if rank != 0:
        finish(world)
        return

    peaks = measured_peaks()
    ms_step = ms_total / args.steps
    fps = N / (n_steps * ms_step / 1e3)
    if ms_e2e == ms_e2e:                                  # not NaN: the host-buffer leg ran
        ms_step_e2e = round(ms_e2e / args.steps, 3)
        fps_e2e = round(N / (n_steps * ms_step_e2e / 1e3), 4)
    else:                                                 # --skip-e2e (profiling runs)
        ms_step_e2e = fps_e2e = None
    lat_bytes = x0.numel() * x0.element_size()

    # dominant hot-path kernel by summed launch time inside the timed region
    roofline = None
    if kernel_times:
        dom = max(kernel_times, key=lambda k_: kernel_times[k_]["ms"])
        kt = kernel_times[dom]
        traffic = None
        tpath = os.path.join(REPO, "profiles", "roofline_traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                traffic = json.load(f).get(dom)
        if dom in TENSOR_KERNELS:
            achieved = kt["work"] / (kt["ms"] * 1e-3) / 1e12
            roofline = {"kernel": dom, "bound": "tensor", "achieved": round(achieved, 2), "peak": peaks["tf_sustained"],
                        "unit": "TFLOP/s", "frac": round(achieved / peaks["tf_sustained"], 4), "traffic": traffic,
                        "peak_source": f"{peaks['source']} sustained cuBLAS bf16 (kernel timed inside a long step)"}
        else:
            achieved = kt["work"] / (kt["ms"] * 1e-3) / 1e9
            roofline = {"kernel": dom, "bound": "hbm", "achieved": round(achieved, 1), "peak": peaks["hbm_gbs"],
                        "unit": "GB/s", "frac": round(achieved / peaks["hbm_gbs"], 4), "traffic": traffic,
                        "peak_source": f"{peaks['source']} HBM copy"}
        roofline["launches"] = kt["launches"]
        roofline["avg_launch_ms"] = round(kt["ms"] / max(1, kt["launches"]), 4)
        roofline["timing"] = ("event-record nodes inside the captured step graph, last replay of the timed region"
                              if args.graph else "CUDA events around every launch in the timed region") + \
                             ("; slowest rank per kernel" if world > 1 else "")
    per_kernel = {}
    for name, kt in kernel_times.items():
        rate = kt["work"] / (kt["ms"] * 1e-3) if kt["ms"] > 0 else 0.0
        ent = {"launches_per_step": int(round(kt["launches"] / per_step_div)), "ms_per_step": round(kt["ms"] / per_step_div, 3),
               ("tflops" if name in TENSOR_KERNELS else "gbs"): round(rate / (1e12 if name in TENSOR_KERNELS else 1e9), 2)}
        if "ms_min_rank" in kt:
            ent["ms_per_step_min_rank"] = round(kt["ms_min_rank"] / per_step_div, 3)
            ent["ms_per_step_rank0"] = round(kt_rank0.get(name, {}).get("ms", 0.0) / per_step_div, 3)
        per_kernel[name] = ent

    cpu = cpu_baseline_sample(cfg_name, args.cpu_threads) if (world == 1 and not args.no_cpu_baseline) else None

    line = {
        "metric": metric_name(cfg_name), "value": round(fps, 4), "unit": "frames/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_step, 3), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "fp16", "data": "synthetic",
        "config": {"workload": workload(cfg_name), "name": cfg_name, "n_frames": N, "keyframes": N // c["batch"],
                   "denoising_steps": n_steps,
                   "frames_per_sec_definition": f"n_frames / ({n_steps} * mean denoising-step time over the timed steps)",
                   "parallelism": f"frames sharded over {world} GPU(s)" if world > 1 else "single GPU",
                   "frames_per_pass": (N // world) if (world > 1 or args.fused_pass) else args.frames_per_pass,
                   "unet_calls_per_step": 1 if args.fused_pass else (2 if world > 1 else 1 + -(-N // (args.frames_per_pass or N))),
                   "cuda_graph": bool(args.graph),
                   "schedule": ("dual-stream: pivotal pass on a side stream under the frame pass, per-block events"
                                if ed.config.get("dual_stream")
                                else "fused: pivotal + frame samples in one UNet call"),
                   "collectives": ("tf_allgather (C ABI, NCCL)" if comm is not None else
                                                                   ("torch.distributed" if world > 1 else None)),
                   "l2": "inputs > L2: every step streams ~10 GB of activations through the UNet (no flush needed)"},
        "e2e": {"value": fps_e2e, "unit": "frames/s", "ms_per_step": ms_step_e2e,
                "h2d_bytes_per_step": 2 * lat_bytes, "d2h_bytes_per_step": lat_bytes},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "roofline": roofline,
        "kernels": per_kernel,
        "hot_path_ms_per_step": round(sum(k_["ms"] for k_ in kernel_times.values()) / per_step_div, 3),
        "finite": finite,
    }
    if verify is not None:
        line["verify"] = verify
    if gpu_ref is not None:
        line["gpu_reference"] = gpu_ref
    if cpu is not None:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)
    finish(world)


def finish(world):
    """End of a rank's run.  With several ranks the process leaves through os._exit after a final barrier: captured
    CUDA graphs still reference the NCCL communicators, and tearing those down in interpreter-exit order can block
    (a 2-rank run with graph-captured torch.distributed collectives hung in destroy_process_group this round)."""
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        try:
            torch.cuda.synchronize()
            torch.distributed.barrier()
        finally:
            os._exit(0)


# ------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's algorithm (oracle port) on the host cores
# ------------------------------------------------------------------------------------------------
def unet_levels(kind, latent):
    """(S, dim, heads, blocks) of the four attention resolutions of the SD UNet at this latent size."""
    from tokenflow_b200 import sd_unet
    cfg = {"sd15": sd_unet.sd15_config, "sd21": sd_unet.sd21_config, "tiny": sd_unet.tiny_config}[kind]()
    ch, heads = cfg.block_out_channels, cfg.num_heads
    s0 = latent * latent
    return ((s0, ch[0], heads[0], 5), (s0 // 4, ch[1], heads[1], 5), (s0 // 16, ch[2], heads[2], 5), (s0 // 64, ch[3], heads[3], 1))


def pick_cpu_threads(requested=None):
    """Host threads for the CPU arm.  BASELINE.md §3 says all cores; on the many-core GPU hosts the oracle's eager
    PyTorch ops get SLOWER past a few dozen threads (128 threads: 15x slower than 32 on this pool), so unless
    --cpu-threads is given a short probe (one SD-sized conv + GEMM) picks the fastest of {all, 1/2, 1/4, 32, 16} cores.
    Returns (threads, {candidate: probe_ms})."""
    ncpu = os.cpu_count() or 1
    if requested:
        return int(requested), {}
    cands = sorted({c for c in (ncpu, ncpu // 2, ncpu // 4, 32, 16) if 1 <= c <= ncpu}, reverse=True)
    if len(cands) == 1:
        return cands[0], {}
    x = torch.randn(3, 320, 64, 64)
    w = torch.randn(320, 320, 3, 3)
    a, b = torch.randn(4096, 320), torch.randn(320, 4096)
    probe = {}
    with torch.no_grad():
        for c in cands:
            torch.set_num_threads(c)
            torch.nn.functional.conv2d(x, w, padding=1); a @ b                     # warm-up at this thread count
            t0 = time.perf_counter()
            for _ in range(2):
                torch.nn.functional.conv2d(x, w, padding=1)
                a @ b
            probe[c] = round((time.perf_counter() - t0) * 500.0, 2)
    best = min(probe, key=probe.get)
    return best, probe


class CpuSampler:
    """Bounded samples of one denoising step of the configured workload on the host cores (fp32) — the
    reference's algorithm through the oracle port.

    The full C2 step is ~20 minutes on 8 cores (135 UNet sample-forwards + ~11 TFLOP of hot path), so each
    sample measures the step's pieces at full resolution and composes them with the exact op counts:
      body   : one frame pass of ONE frame (3 stream samples) through the hooked UNet with the oracle ops;
               per-sample body time x 3*(K+N) sample-forwards per step
      nn/prop: the NN field of that frame against one keyframe and its propagation, timed inside the body
               pass, x the config's counts (2N-B frame/keyframe pairs, N frames)
      attn   : `oracle.extended_attention` (the restated reference closure, tokenflow_utils.py:114-199) for ONE
               head of a K-keyframe pivotal pass at each of the 4 UNet levels; x heads x blocks
    The result is therefore EXTRAPOLATED from a bounded sample (marked so in the JSON)."""

    def __init__(self, kind="sd15", latent=64, ctx_dim=None, levels=None, n_frames=40, batch=8, n_timesteps=50,
                 n_steps=50, mode="pnp", threads=None, attn_keyframes=None):
        from oracle.oracle_ops import OracleOps
        from tokenflow_b200 import sd_unet, tokenflow_utils as tfu
        from tokenflow_b200.editor import TokenFlowEditor, synthetic_inputs
        from tokenflow_b200.scheduler import DDIMScheduler
        self.threads, self.thread_probe = pick_cpu_threads(threads)
        torch.set_num_threads(self.threads)
        self.tfu = tfu
        self.N, self.B, self.n_steps = n_frames, batch, n_steps
        self.K = n_frames // batch
        self.attn_K = attn_keyframes or self.K

        class TimedOracle(OracleOps):
            def __init__(self):
                self.t = {"nn": 0.0, "prop": 0.0}

            def nn_field(self, *a, **k):
                t0 = time.perf_counter(); r = super().nn_field(*a, **k); self.t["nn"] += time.perf_counter() - t0; return r

            def propagate(self, *a, **k):
                t0 = time.perf_counter(); r = super().propagate(*a, **k); self.t["prop"] += time.perf_counter() - t0; return r

        self.ops = TimedOracle()
        tfu._install_ops_for_testing(self.ops)
        with torch.no_grad():
            self.levels = levels or unet_levels(kind, latent)
            unet = sd_unet.build_unet(kind, seed=1)
            ctx_dim = ctx_dim or unet.config.cross_attention_dim
            cfg = {"n_frames": 1, "batch_size": 1, "n_timesteps": n_timesteps, "guidance_scale": 7.5, "mode": mode}
            self.x, text, pnp, src = synthetic_inputs(1, latent, ctx_dim, n_timesteps, seed=1)
            self.ed = TokenFlowEditor(unet, DDIMScheduler(), tfu, cfg, text, pnp, source_latents=lambda t: src[t])
            self.ed.init_method()
            self.t0 = self.ed._t_host[0]
            tfu.register_pivotal(self.ed, True)
            self.ed.denoise_step(self.x, self.t0, torch.arange(1))      # fills the caches (K=1), untimed
            tfu.register_pivotal(self.ed, False)
            tfu.register_batch_idx(self.ed, 0)
        tfu._install_ops_for_testing(None)

    def step(self):
        from oracle import tokenflow_oracle as O
        K, N, B = self.K, self.N, self.B
        self.tfu._install_ops_for_testing(self.ops)
        try:
            with torch.no_grad():
                self.ops.t = {"nn": 0.0, "prop": 0.0}
                t0 = time.perf_counter()
                self.ed.denoise_step(self.x, self.t0, torch.arange(1))  # 3 sample-forwards + NN(1 pair) + propagate(1 frame)
                t_pass = time.perf_counter() - t0
                t_nn_pair, t_prop_frame = self.ops.t["nn"], self.ops.t["prop"]
                t_body_sample = (t_pass - t_nn_pair - t_prop_frame) / 3.0
                t_attn = 0.0
                ka = self.attn_K
                for S, dim, heads, blocks in self.levels:
                    d = dim // heads
                    q, k, v = (torch.randn(3 * ka, S, d) for _ in range(3))
                    t0 = time.perf_counter()
                    O.extended_attention(q, k, v, 1, d ** -0.5, False)      # one head of a K-keyframe pivotal pass
                    # scaled to the config's K when the sample uses fewer keyframes (cost ~ K*(2K+1))
                    t_attn += (time.perf_counter() - t0) * heads * blocks * (K * (2 * K + 1)) / (ka * (2 * ka + 1))
        finally:
            self.tfu._install_ops_for_testing(None)
        n_body, n_pairs = 3 * (K + N), 2 * N - B
        t_step = t_body_sample * n_body + t_attn + t_nn_pair * n_pairs + t_prop_frame * N
        desc = ("per step: one full-resolution frame pass (3 UNet sample-forwards + NN field vs 1 keyframe + propagation) and "
                f"oracle.extended_attention for one head of a K={ka} pivotal pass per UNet level, fp32, composed with the "
                f"config's op counts (body {t_body_sample:.2f}s/sample x{n_body}, attn {t_attn:.1f}s, nn {t_nn_pair:.2f}s/pair "
                f"x{n_pairs}, prop {t_prop_frame:.3f}s/frame x{N})")
        return t_step, desc


def make_sampler(cfg_name, threads=None):
    c = CONFIGS[cfg_name]
    K = c["n_frames"] // c["batch"]
    return CpuSampler(kind=c["kind"], latent=c["latent"], n_frames=c["n_frames"], batch=c["batch"], n_timesteps=c["n_timesteps"],
                      n_steps=c["n_steps"], mode=c["mode"], threads=threads, attn_keyframes=min(K, 5))


def cpu_baseline_sample(cfg_name="C2", threads=None):
    c = CONFIGS[cfg_name]
    sampler = make_sampler(cfg_name, threads)
    t_step, desc = sampler.step()
    return {"value": round(c["n_frames"] / (c["n_steps"] * t_step), 6), "unit": "frames/s", "cores": torch.get_num_threads(),
            "host_cpus": os.cpu_count(), "threads_probe_ms": getattr(sampler, "thread_probe", {}), "kind": "port",
            "extrapolated": True, "sample": desc, "s_per_step_extrapolated": round(t_step, 2)}


def run_reference(args):
    rank, _, world = dist_env()
    if rank != 0:
        return
    cfg_name = getattr(args, "config", "C2")
    c = CONFIGS[cfg_name]
    sampler = make_sampler(cfg_name, getattr(args, "cpu_threads", None)) if CpuSampler is _REAL_SAMPLER else CpuSampler()
    times, desc = [], ""
    for i in range(args.warmup + args.steps):
        t_step, desc = sampler.step()
        if i >= args.warmup:
            times.append(t_step)
    t_step = sum(times) / len(times)
    fps = c["n_frames"] / (c["n_steps"] * t_step)
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": metric_name(cfg_name), "value": round(fps, 6), "unit": "frames/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(t_step * 1e3, 1), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "fp32", "data": "synthetic", "extrapolated": True,
            "config": {"workload": workload(cfg_name), "name": cfg_name,
                       "note": "reference algorithm (oracle port) on host cores; each step is a bounded sample of the "
                               "step composed with exact op counts: the value is EXTRAPOLATED, not a full run"},
            "cpu_baseline": {"value": round(fps, 6), "unit": "frames/s", "cores": cores, "host_cpus": os.cpu_count(),
                             "threads_probe_ms": getattr(sampler, "thread_probe", {}), "kind": "port",
                             "extrapolated": True, "sample": desc},
            "e2e": {"value": round(fps, 6), "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


_REAL_SAMPLER = CpuSampler


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="C2", choices=sorted(CONFIGS), help="BASELINE.json workload (default C2)")
    ap.add_argument("--verify", action="store_true",
                    help="before timing: 2 steps of the measured path vs the 1-rank eager path (max |diff|, NN-index mismatches)")
    ap.add_argument("--graph", type=int, default=1, help="1: replay the fused step as a CUDA graph (default); 0: eager")
    ap.add_argument("--dual-stream", type=int, default=-1,
                    help="1: pivotal pass on a side stream concurrent with the frame pass (experimental: slower on one GPU, "
                         "not validated with NCCL ranks); 0 / -1 (default): one fused UNet call per step")
    ap.add_argument("--no-kernel-events", action="store_true", help="capture / run without per-launch timing events")
    ap.add_argument("--torch-collectives", action="store_true", help="all-gathers through torch.distributed instead of the C ABI")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-threads", type=int, default=None, help="host threads of the CPU arm (default: os.cpu_count())")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--gpu-reference-steps", type=int, default=2, help="steps of the reference-GPU-arithmetic leg (N=1 only)")
    ap.add_argument("--skip-e2e", action="store_true", help="profiling runs only: skip the host-buffer leg")
    ap.add_argument("--no-channels-last", action="store_true", help="UNet body in NCHW instead of channels_last")
    ap.add_argument("--frames-per-pass", type=int, default=None,
                    help="frames per frame-pass UNet call when --fused-pass 0 (8 = the reference's per-batch schedule; "
                         "default: all frames of the GPU in one pass with per-frame keyframe tables — identical results)")
    ap.add_argument("--fused-pass", type=int, default=1,
                    help="1: one UNet call per step and GPU ([pivotal samples | frames], keyframe caches filled and "
                         "consumed inside each block); 0: the reference's pivotal pass + frame passes")
    ap.add_argument("--cudnn-benchmark", type=int, default=1, help="torch.backends.cudnn.benchmark for the UNet body convs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the latents the last timed step returned as DIR/latents.npy "
                         "(float32; the inputs depend only on the arguments)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs --impl ours: the reference arm times samples of a step and returns no latents")
    if not args.fused_pass:
        args.graph = 0                                   # graphs capture the fused step only
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
