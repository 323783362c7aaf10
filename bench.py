#!/usr/bin/env python
"""bench.py -- Diffuman4D window denoise-steps/sec on B200 (BASELINE.json metric).

A "step" is ONE window denoise step of the reference's sliding-window sampler
(pipeline_diffuman4d.py:369-425): input assembly -> UNet forward on 2F images (CFG) -> CFG combine -> F per-frame
DDIM updates.  Workload at N=1: the spatial window W16 of `demo_4d_tiny` (4 cond + 12 target frames, CFG => 32
images, SD-2.1 layout UNet, latents 64x64 -- BASELINE's synthetic size).  Synthetic seeded inputs, random-init
weights of the real architecture (no network for the checkpoint).

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...   (weak scaling: every
        rank denoises its own window; windows of one sampler round are independent units, SURVEY.md section 8e.1;
        the line also carries a `sharded` object: ONE window frame-sharded over the N ranks, SURVEY 8e.2)
    python bench.py --impl reference ...   (the CPU oracle -- the reference's torch graph restated -- on host cores,
        REAL W16 window steps, as many of the requested --steps as fit the time budget)

Everything printed is measured in this run; figures that come from a committed profile name the file they were read from.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import re
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = dict(name="demo_4d_tiny spatial window W16 (4 cond + 12 target frames), CFG 2.0, latents 64x64",
                F=16, n_cond=4, h=64, w=64, guidance=2.0, domain="spatial", n_steps=18)
# other BASELINE configurations, timed at N=1 as `also` entries (not the headline)
ALSO = [dict(key="W24_temporal_64", name="temporal window W24 (12 cond + 12 target frames), CFG 2.0, latents 64x64",
             F=24, n_cond=12, h=64, w=64, domain="temporal", steps=5),
        dict(key="W16_spatial_128", name="spatial window W16, CFG 2.0, latents 128x128 (reference default, 1024^2 px)",
             F=16, n_cond=4, h=128, w=128, domain="spatial", steps=3)]
METRIC = "unet_window_denoise_steps_per_sec"
UNIT = "window-steps/s"
# ncu --set full capture of the dominant kernel (tools/gpu_profile.sh -> tools/ncu_summary.py); parsed at run time
NCU_SUMMARIES = ["profiles/r02_ncu_attention.txt", "profiles/r01d_ncu_attention.txt"]


def synth_inputs(F, n_cond, h, w, pose=True, seed=0):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g)
    d = dict(latents=r(F, 4, h, w), pixel=r(F, 4, h, w), plucker=(torch.rand(F, 6, h, w, generator=g) * 2 - 1),
             mask=torch.ones(F, 1, h, w))
    d["mask"][:n_cond] = 0
    d["skel"] = (torch.rand(F, 3, 8 * h, 8 * w, generator=g) * 2 - 1) if pose else r(F, 4, h, w)
    ti = torch.zeros(F, dtype=torch.int64)
    tgt = F - n_cond
    ti[n_cond:] = torch.tensor([min(17, (tgt - 1 - i) // 2) for i in range(tgt)])   # staggered like PIPE:503-543
    d["ts"] = ti
    return d


class ClockSampler(threading.Thread):
    FIELDS = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self._halt = index, [], threading.Event()

    def run(self):
        while not self._halt.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}",
                                    "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                p = [x.strip() for x in o.strip().split(",")]
                if len(p) >= 6:
                    self.samples.append(p)
            except Exception:  # noqa: BLE001
                pass
            self._halt.wait(0.2)

    def stop(self):
        self._halt.set()
        self.join(timeout=3)
        sm = sorted(int(s[0]) for s in self.samples if s[0].isdigit())
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(s[2 + i].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.samples)}


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel, read from the newest committed ncu summary
    (never a literal): returns (bytes, file) or (None, None)."""
    for rel in NCU_SUMMARIES:
        path = os.path.join(ROOT, rel)
        if not os.path.exists(path):
            continue
        tot, found = 0.0, 0
        for line in open(path):
            m = re.match(r"\s*dram__bytes_(read|write)\.sum\s+([0-9.]+)\s+(\w+)", line)
            if m and found < 2:   # first kernel block of the file
                mult = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}.get(m.group(3), 1.0)
                tot += float(m.group(2)) * mult
                found += 1
        if found == 2:
            return int(tot), rel
    return None, None


# ------------------------------------------------------------------------------------------------------- CPU arm
def calibrate_cpu_threads():
    """Pick the torch thread count that maximises fp32 conv throughput on this host (a cgroup-limited box can be much
    slower with one thread per visible core).  Returns (threads, conv GFLOP/s)."""
    import torch.nn.functional as Fn
    try:
        usable = len(os.sched_getaffinity(0))
    except AttributeError:
        usable = os.cpu_count() or 1
    x = torch.randn(4, 320, 64, 64)
    wgt = torch.randn(320, 320, 3, 3)
    fl = 2.0 * 4 * 64 * 64 * 320 * 320 * 9
    best = (1, 0.0)
    for nt in sorted({usable, max(1, usable // 2), max(1, usable // 4), min(usable, 16), min(usable, 8)}):
        torch.set_num_threads(nt)
        Fn.conv2d(x, wgt, padding=1)
        t0 = time.perf_counter()
        for _ in range(2):
            Fn.conv2d(x, wgt, padding=1)
        g = 2 * fl / (time.perf_counter() - t0) / 1e9
        if g > best[1]:
            best = (nt, g)
    torch.set_num_threads(best[0])
    return best


def cpu_oracle_w16_steps(max_steps: int, budget_s: float):
    """Times the oracle (test infrastructure, used here ONLY as the reported CPU baseline) on REAL window steps of the
    benchmark workload (W16 @ 64x64, 32 images, 31.94 TFLOP each): as many of ``max_steps`` as fit ``budget_s`` after the
    first one, never fewer than one.  No FLOP scaling.  Returns (seconds per step list, threads)."""
    from diffuman4d_b200.config import SchedulerConfig, UNetConfig
    from diffuman4d_b200.weights import random_state_dict
    from oracle.pipeline_oracle import DDIMOracle, denoise_window_oracle
    from oracle.unet_oracle import OracleUNet
    threads, _ = calibrate_cpu_threads()
    cfg = UNetConfig.sd21()
    wl = WORKLOAD
    net = OracleUNet(cfg).eval()
    net.load_state_dict({k: v.float() for k, v in random_state_dict(cfg, seed=1).items()})
    d = synth_inputs(wl["F"], wl["n_cond"], wl["h"], wl["w"])
    sched = DDIMOracle(SchedulerConfig())
    sched.set_timesteps(wl["n_steps"])

    def unet(x, t, sk, doms, nf):
        with torch.no_grad():
            return net(x, t, sk, doms, nf)

    times = []
    t_start = time.perf_counter()
    while len(times) < max(1, max_steps):
        t0 = time.perf_counter()
        denoise_window_oracle(unet, sched, latents=d["latents"].clone(), pixel_latents=d["pixel"], plucker=d["plucker"],
                              skeletons=d["skel"], cond_mask=d["mask"], timestep_indices=d["ts"], domain=wl["domain"],
                              guidance_scale=wl["guidance"])
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start + times[-1] > budget_s:
            break
    return times, threads


def cpu_baseline_obj(times, threads, requested):
    from diffuman4d_b200.config import UNetConfig
    from diffuman4d_b200.flops import unet_flops
    wl = WORKLOAD
    fl = unet_flops(UNetConfig.sd21(), 2 * wl["F"], wl["F"], wl["h"], wl["w"])["total"]
    sec = sum(times) / len(times)
    return {"value": 1.0 / sec, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": (f"oracle (fp32 torch restatement of the reference graph; diffusers itself is not installable here): "
                       f"{len(times)} REAL W16@64x64 window step(s) of {requested} requested, {fl / 1e12:.2f} TFLOP each, "
                       f"{sec:.2f} s/step on {threads} torch threads (calibrated); no FLOP scaling"),
            "steps_timed": len(times), "same_config": True, "gflops": fl / sec / 1e9}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    t0 = time.perf_counter()
    times, threads = cpu_oracle_w16_steps(args.steps, budget_s=170.0)
    cb = cpu_baseline_obj(times, threads, args.steps)
    val = cb["value"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 / val, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD["name"],
                   "note": "CPU-port baseline: the oracle's torch graph (the reference's graph restated; diffusers is not "
                           "installable here) on the host cores, full W16 window steps; NOT the upstream bf16-GPU pipeline",
                   "steps_timed": len(times)},
        "cpu_baseline": cb, "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0}))


# ------------------------------------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch.distributed as dist
    from diffuman4d_b200 import build as d4d_build
    from diffuman4d_b200._lib import check, lib
    from diffuman4d_b200.config import SchedulerConfig, UNetConfig
    from diffuman4d_b200.flops import unet_flops
    from diffuman4d_b200.pipeline import B200Diffuman4DPipeline
    from diffuman4d_b200.unet import B200MultiviewUNet
    from diffuman4d_b200.weights import random_state_dict

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a B200: there is no CPU fallback for the product path")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    if not os.path.exists(os.path.join(ROOT, "diffuman4d_b200", "libd4d.so")):
        d4d_build.build(test_lib=False)
    dev = torch.device("cuda", local)
    cfg = UNetConfig.sd21()
    wl = WORKLOAD
    F, h, w = wl["F"], wl["h"], wl["w"]
    sd = random_state_dict(cfg, seed=1)
    unet = B200MultiviewUNet(cfg, local).load_state_dict(sd)
    pipe = B200Diffuman4DPipeline(unet, SchedulerConfig())
    pipe.parepare_schedulers(wl["n_steps"], F)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    peak_tf = peaks.get("bf16_tflops_sustained", 1400.0)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        barrier()
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    def make_stepper(p, inputs, domain, shard=None, F_total=None):
        """Resident-input window step: restores latents / indices from device copies, then ONE public denoise_window call."""
        devt = {k: (v.to(torch.bfloat16) if v.dtype.is_floating_point else v).to(dev) for k, v in inputs.items()}
        lat, ts = devt["latents"].clone(), devt["ts"].clone()

        def step():
            lat.copy_(devt["latents"])
            ts.copy_(devt["ts"])
            kw = dict(latents=lat, pixel_values_latents=devt["pixel"], plucker_embeds_latents=devt["plucker"],
                      skeletons_latents=devt["skel"], cond_masks_latents=devt["mask"], timestep_indices=ts, domain=domain,
                      guidance_scale=wl["guidance"])
            if shard is not None:
                shard.denoise_window(F_total=F_total, **kw)
            else:
                p.denoise_window(**kw)
        return step, lat, ts

    # ================= headline: replicas (N=1: the single window) =================
    full_inputs = synth_inputs(F, wl["n_cond"], h, w, seed=rank)
    host = {k: (v.to(torch.bfloat16) if v.dtype.is_floating_point else v).pin_memory() for k, v in full_inputs.items()}
    step_resident, lat_res, ts_res = make_stepper(pipe, full_inputs, wl["domain"])

    out_host = torch.empty_like(host["latents"]).pin_memory()
    ts_host = torch.empty_like(host["ts"]).pin_memory()
    # e2e = the public call fed from pinned HOST buffers: every step uploads its own inputs (H2D) and reads its result
    # back (D2H).  The upload of step i+1 is issued on a copy stream while step i computes (double-buffered staging), as
    # a caller streaming windows through the pipeline would do; each step still ends with a stream synchronisation.
    stages = [{k: torch.empty_like(v, device=dev) for k, v in host.items()} for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    h2d_done = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_state = {"i": 0, "primed": False}
    KEYS = ("latents", "pixel", "plucker", "skel", "mask", "ts")

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            for k in KEYS:
                stages[slot][k].copy_(host[k], non_blocking=True)
            h2d_done[slot].record(copy_stream)

    def step_e2e():
        i = e2e_state["i"]
        cur = i & 1
        if not e2e_state["primed"]:
            upload(cur)
            e2e_state["primed"] = True
        upload(cur ^ 1)                                   # inputs of the NEXT step, overlapped with this step's compute
        torch.cuda.current_stream().wait_event(h2d_done[cur])
        st = stages[cur]
        pipe.denoise_window(latents=st["latents"], pixel_values_latents=st["pixel"], plucker_embeds_latents=st["plucker"],
                            skeletons_latents=st["skel"], cond_masks_latents=st["mask"], timestep_indices=st["ts"],
                            domain=wl["domain"], guidance_scale=wl["guidance"])
        out_host.copy_(st["latents"], non_blocking=True)
        ts_host.copy_(st["ts"], non_blocking=True)
        torch.cuda.current_stream().synchronize()
        e2e_state["i"] = i + 1

    sampler = ClockSampler(local)
    sampler.start()
    ms_res = timed(step_resident, args.steps, max(args.warmup, 3))
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # what denoise_window hands back to its caller after the last timed step: the window's latents and timestep
        # indices, both updated in place
        dump_outputs(args.dump_outputs, {"latents": lat_res.float().cpu().numpy(),
                                         "timestep_indices": ts_res.cpu().double().numpy()})
    ms_e2e = timed(step_e2e, args.steps, 1)
    assert torch.isfinite(out_host.float()).all(), "non-finite latents out of the window step"

    # ---- live per-kernel-kind device times of the UNet forward (CUDA events around every launch; N=1 plan) ----
    B = 2 * F
    x = torch.randn(B, cfg.in_channels, h, w, device=dev).to(torch.bfloat16)
    tt = torch.randint(0, 1000, (B,), device=dev)
    skp = torch.rand(F, 3, 8 * h, 8 * w, device=dev).to(torch.bfloat16) * 2 - 1
    sk = torch.cat([-torch.ones_like(skp), skp])
    y = torch.empty(B, 4, h, w, device=dev, dtype=torch.bfloat16)
    doms = (C.c_int32 * 2)(0, 0)
    ms_k, n_k, fl_k = (C.c_float * 6)(), (C.c_int32 * 6)(), (C.c_double * 6)()
    acc = [0.0] * 6
    reps = 3
    for i in range(reps + 1):
        check(lib().d4d_profile_forward(unet._h, x.data_ptr(), tt.data_ptr(), sk.data_ptr(), doms, 2, B, F, h, w,
                                        y.data_ptr(), torch.cuda.current_stream().cuda_stream, ms_k, n_k, fl_k))
        if i > 0:
            acc = [a + m for a, m in zip(acc, ms_k)]
    kind_ms = [a / reps for a in acc]
    del x, skp, sk, y
    fl = unet_flops(cfg, B, F, h, w)
    alg = {0: fl["linear"] + fl["ff"], 1: fl["conv3x3"], 2: fl["attn3d"] + fl["attn2d"]}
    names = ["gemm", "conv3x3", "attention", "groupnorm", "layernorm", "other"]
    top = max((0, 1, 2), key=lambda k: kind_ms[k])
    achieved = alg[top] / (kind_ms[top] * 1e-3) / 1e12
    launches_fwd = unet.forward_launches(2, B, F, h, w)
    launches_step = launches_fwd + 3   # + assemble, cfg-skeleton, cfg+ddim kernels (2 memcpys not counted)
    traffic, traffic_file = (ncu_traffic() if (world == 1 and names[top] == "attention") else (None, None))
    roofline = {"bound": "tensor", "kernel": names[top], "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                "frac": achieved / peak_tf,
                "traffic": traffic,
                "traffic_note": (f"dram__bytes_read.sum + dram__bytes_write.sum of ONE captured launch, parsed at run time from "
                                 f"{traffic_file} (ncu --set full); not re-measured in this run" if traffic_file else
                                 "no ncu capture consulted in this run"),
                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback 1.4 PFLOP/s sustained",
                "launches_per_forward": int(n_k[top]), "ms_per_forward": kind_ms[top],
                "by_kind_ms": {names[k]: round(kind_ms[k], 4) for k in range(6)},
                "by_kind_tflops": {names[k]: round(alg[k] / (kind_ms[k] * 1e-3) / 1e12, 1) for k in (0, 1, 2)},
                "by_kind_note": "one UNet forward of the single-GPU W16 plan with the 2F-image pose batch (the window step shares "
                                "the CFG-negative pose embedding: F+1 images)",
                "unet_forward_ms_sum": round(sum(kind_ms), 3)}

    value = world * args.steps / (ms_res * 1e-3)
    e2e_val = world * args.steps / (ms_e2e * 1e-3)
    h2d = sum(host[k].numel() * host[k].element_size() for k in KEYS)
    d2h = out_host.numel() * 2 + ts_host.numel() * 8
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": ms_res / args.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": wl["name"], "unet": "SD-2.1 layout 320/640/1280/1280, heads 5/10/20/20, in_channels 11 "
                   "(pose encoder + frame-index embedding), no attn2", "images_per_step": B,
                   "parallelism": (f"replicas x{world} (independent windows, no collective)" if world > 1 else "single GPU"),
                   "l2": f"no explicit flush: one step streams ~{unet.workspace_bytes(2, B, F, h, w) / 2**30:.1f} GiB of "
                         "activations + 1.6 GB of weights through a 126 MB L2"},
        "tflops_per_step": fl["total"] / 1e12,
        "unet_tflops_achieved": fl["total"] / (ms_res / args.steps * 1e-3) / 1e12,
        "unet_roofline_frac": fl["total"] / (ms_res / args.steps * 1e-3) / 1e12 / peak_tf,
        "roofline": roofline, "clocks": clocks,
        "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches_step * args.steps,
    }

    # ================= N > 1: the same window frame-sharded over all ranks (north-star split, SURVEY 8e.2) =================
    if world > 1 and F % world == 0 and not args.no_sharded:
        try:
            from diffuman4d_b200.sharded import FrameShardedPipeline
            shared = synth_inputs(F, wl["n_cond"], h, w, seed=0)          # every rank: the SAME window
            # single-GPU result of that window on this rank (bit-identity reference for this rank's frames)
            step_single, lat_single, ts_single = make_stepper(pipe, shared, wl["domain"])
            step_single()
            torch.cuda.synchronize()
            sh = FrameShardedPipeline(pipe, max_frames=F, h=h, w=w)
            lo, hi = sh.frames(F)
            step_sh, lat_sh, ts_sh = make_stepper(pipe, {k: v[lo:hi].contiguous() for k, v in shared.items()}, wl["domain"],
                                                  shard=sh, F_total=F)
            ssteps = args.steps
            ms_sh = timed(step_sh, ssteps, 3)
            same = torch.equal(lat_sh, lat_single[lo:hi]) and torch.equal(ts_sh, ts_single[lo:hi])
            flag = torch.tensor([1 if same else 0], device=dev)
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
            line["sharded"] = {
                "what": f"ONE W16 window per step, frames split over {world} ranks ({F // world} frames = {2 * F // world} images per rank), "
                        "K/V of the 11 3-D attention layers exchanged over NVLink peer memory inside the QKV GEMM epilogue",
                "value": ssteps / (ms_sh * 1e-3), "unit": UNIT, "ms_per_window": ms_sh / ssteps, "scaling": "strong",
                "speedup_vs_this_runs_single_gpu_step": (ms_res / args.steps) / (ms_sh / ssteps),
                "bit_identical_to_single_gpu": bool(flag.item()),
                "unet_roofline_frac_per_gpu": fl["total"] / (ms_sh / ssteps * 1e-3) / 1e12 / peak_tf / world}
        except Exception as e:  # noqa: BLE001 -- the replicas line above is already measured: report it even if this extra fails
            line["sharded"] = {"error": str(e)[:300]}
            if rank == 0:
                print(json.dumps(line), flush=True)
            os._exit(0)   # the process group / CUDA context may be unusable: do not hang in its teardown

    # ================= N = 1 extras: other BASELINE configurations, GPU-eager and CPU baselines =================
    if world == 1 and not args.quick:
        also = {}
        for a in ALSO:
            try:
                Fa, ha, wa = a["F"], a["h"], a["w"]
                pipe.parepare_schedulers(wl["n_steps"], Fa)
                stp, _, _ = make_stepper(pipe, synth_inputs(Fa, a["n_cond"], ha, wa, seed=1), a["domain"])
                ms_a = timed(stp, a["steps"], 2)
                fa = unet_flops(cfg, 2 * Fa, Fa, ha, wa)["total"]
                also[a["key"]] = {"workload": a["name"], "value": a["steps"] / (ms_a * 1e-3), "unit": UNIT,
                                  "ms_per_step": ms_a / a["steps"], "steps": a["steps"], "tflops_per_step": fa / 1e12,
                                  "unet_roofline_frac": fa / (ms_a / a["steps"] * 1e-3) / 1e12 / peak_tf}
                del stp
                torch.cuda.empty_cache()
            except Exception as e:  # noqa: BLE001
                also[a["key"]] = {"error": str(e)[:200]}
        line["also"] = also
        pipe.parepare_schedulers(wl["n_steps"], F)
        if not args.no_eager_baseline:
            line["gpu_eager_bf16_baseline"] = gpu_eager_baseline(cfg, sd, full_inputs, dev, args.steps)
        if not args.no_cpu_baseline:
            times, threads = cpu_oracle_w16_steps(1, budget_s=30.0)
            line["cpu_baseline"] = cpu_baseline_obj(times, threads, 1)
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """Writes every array as ``out_dir/<name>.npy``, so two builds run with the same arguments (hence the same seeded
    inputs and weights) can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


def gpu_eager_baseline(cfg, sd, inputs, dev, steps):
    """The same window step as the reference would execute it on THIS GPU: the oracle's torch graph in bf16 on
    cuDNN / cuBLAS / SDPA (eager).  A reported comparator like cpu_baseline -- never part of the product path."""
    from diffuman4d_b200.config import SchedulerConfig
    from oracle.pipeline_oracle import DDIMOracle, denoise_window_oracle
    from oracle.unet_oracle import OracleUNet
    try:
        net = OracleUNet(cfg).eval()
        net.load_state_dict({k: v.float() for k, v in sd.items()})
        net = net.to(dev).to(torch.bfloat16)
        sched = DDIMOracle(SchedulerConfig())
        sched.set_timesteps(WORKLOAD["n_steps"])
        d = {k: (v.to(torch.bfloat16) if v.dtype.is_floating_point else v).to(dev) for k, v in inputs.items()}
        sched.timesteps = sched.timesteps.to(dev)

        def unet(x, t, sk, doms, nf):
            with torch.no_grad():
                return net(x, t, sk, doms, nf)

        def step():
            denoise_window_oracle(unet, sched, latents=d["latents"].clone(), pixel_latents=d["pixel"], plucker=d["plucker"],
                                  skeletons=d["skel"], cond_mask=d["mask"], timestep_indices=d["ts"], domain=WORKLOAD["domain"],
                                  guidance_scale=WORKLOAD["guidance"])
        n = max(3, min(steps, 10))
        for _ in range(2):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / n
        del net
        torch.cuda.empty_cache()
        return {"value": 1e3 / ms, "unit": UNIT, "ms_per_step": ms, "steps": n,
                "what": "oracle torch graph (the reference's graph restated), bf16 eager on this GPU: cuDNN convs, cuBLAS linears, "
                        "SDPA flash attention, per-frame Python scheduler loop (PIPE:413-423)"}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:300]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-eager-baseline", action="store_true")
    ap.add_argument("--no-sharded", action="store_true", help="N>1: skip the frame-sharded `sharded` object")
    ap.add_argument("--quick", action="store_true", help="N=1: headline only (no `also`, no baselines)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the latents and timestep indices "
                    "of the last headline step (rank 0's window) as DIR/<name>.npy in float32 / float64")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
