#!/usr/bin/env python
"""Headline benchmark: value-map steps/sec (BLIP-2 ITM cosine + ValueMap cone-fuse).

Workload = BASELINE.json configs[1]: one environment per GPU, 640x480 RGB-D, 1000^2 x
0.05 m grid, ViT-g/14 + Q-Former ITC (seeded synthetic weights of the real
architecture: no checkpoint exists offline), weighted-average fusion
(use_max_confidence=False, the policies' setting).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch B] [--dump-outputs DIR]

N > 1 is launched by torchrun (one rank per GPU, env shards, NO step-path collective;
NCCL only for the barrier and the max-over-ranks of the timing).  Prints ONE JSON line.
`--impl reference` times the reference's own CPU algorithm (oracle port: numpy/cv2 value
map restated from vlfm/mapping/value_map.py + fp32 HF BLIP-2 ITC) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FOV = float(np.deg2rad(79.0))
MIN_D, MAX_D = 0.5, 5.0
H, W, G = 480, 640, 1000
PROMPT = "Seems like there is a chair ahead."
NFRAMES = 16
# the SAME string in both arms' config.workload
WORKLOAD = ("configs[1]: BLIP-2 ITC (ViT-g/14 + Q-Former, synthetic weights) + ValueMap cone-fuse, batch=1 env/GPU, "
            "640x480 RGB-D, 1000^2 grid, weighted fusion")


def pin_cpu_threads() -> int:
    """The CPU arm uses the host's cores the same way whatever launched it (torchrun exports OMP_NUM_THREADS=1)."""
    import torch

    n = max(1, min(64, (os.cpu_count() or 2) // 2))
    torch.set_num_threads(n)
    try:
        import cv2

        cv2.setNumThreads(n)
    except Exception:
        pass
    return n


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
            p = json.load(fh)
        return p, "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], None, set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def make_frames(seed: int):
    from vlfm_b200.utils.synthetic import trajectory

    return trajectory(seed, NFRAMES, h=H, w=W, with_rgb=True, bound_m=15.0)


# ------------------------------------------------------------------ CPU reference ----
def cpu_reference(steps: int, warmup: int, budget_s: float, frames, state_dict, dims):
    """The reference's own CPU algorithm for this path: fp32 BLIP-2 ITC + numpy/cv2 value map."""
    import torch

    from oracle.blip2_oracle import Blip2Oracle
    from oracle.value_map_oracle import ValueMapOracle

    pin_cpu_threads()
    orc = Blip2Oracle(dims, state_dict)
    vm = ValueMapOracle(1, size=G, use_max_confidence=False, prims="cv2")
    ids = [101, 3849, 2066, 2045, 2003, 1037, 3242, 3805, 1012, 102]
    times = []
    total = steps + warmup
    t_start = time.perf_counter()
    i = 0
    while i < total:
        f = frames[i % len(frames)]
        t0 = time.perf_counter()
        c = orc.cosine(f.rgb, ids)
        vm.update_map(np.array([c]), f.depth, f.tf, MIN_D, MAX_D, FOV)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
        i += 1
        if time.perf_counter() - t_start > budget_s and len(times) >= 1:
            break
    t = float(np.mean(times))
    return 1.0 / t, len(times), torch.get_num_threads()


def run_reference(args):
    import torch

    from vlfm_b200.vlm.blip2_config import Blip2Dims, random_state_dict

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dims = Blip2Dims()
    sd = random_state_dict(dims, 0)
    frames = make_frames(0)
    sps, n, threads = cpu_reference(args.steps, args.warmup, 240.0, frames, sd, dims)
    line = {
        "impl": "reference", "metric": "value-map steps/sec (ITM+cone-fuse)", "value": sps, "unit": "env-steps/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 / sps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "envs_per_gpu": 1,
                   "note": "CPU arm: ONE process on rank 0 with the thread count below, whatever --gpus says (not multiplied by N)"},
        "cpu_baseline": {"value": sps, "unit": "env-steps/s", "cores": threads, "kind": "port",
                         "sample": f"{n} env-steps timed after {args.warmup} warm-up (fp32 HF BLIP-2 ITC forward + numpy/cv2 value-map oracle)",
                         "host_cpus": os.cpu_count(), "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")},
        "e2e": {"value": sps, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------- GPU arm ----
def run_b200(args):
    import torch
    import torch.distributed as dist

    from vlfm_b200 import _lib
    from vlfm_b200.mapping.value_map import ValueMap, ValueMapBatch
    from vlfm_b200.vlm.blip2_config import Blip2Dims, random_state_dict
    from vlfm_b200.vlm.blip2itm import BLIP2ITM

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, K, Wm = args.batch, args.steps, max(args.warmup, 3)
    dims = Blip2Dims()
    sd = random_state_dict(dims, 0)
    itm = BLIP2ITM(state_dict=sd, dims=dims, max_batch=B, device=dev)
    eng = ValueMapBatch(B, 1, size=G, use_max_confidence=False, device=dev)
    frames_per_env = [make_frames(rank * B + e) for e in range(B)]
    rgb = torch.from_numpy(np.stack([np.stack([fr[i].rgb for fr in frames_per_env]) for i in range(NFRAMES)])).to(dev)
    depth = torch.from_numpy(np.stack([np.stack([fr[i].depth for fr in frames_per_env]) for i in range(NFRAMES)])).to(dev)
    tfs = torch.from_numpy(np.stack([np.stack([fr[i].tf for fr in frames_per_env]) for i in range(NFRAMES)])).to(dev)
    lib = _lib.load()

    def step_device(i):
        j = i % NFRAMES
        cos = itm.cosine_device(rgb[j], PROMPT)
        eng.update(cos.double().view(B, 1), depth[j], tfs[j], MIN_D, MAX_D, FOV)
        return cos

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # kernels per step: count C-ABI launches of one un-graphed pass
    itm.engine.use_graph = False
    n0 = lib.vlfm_launch_count(); step_device(0); torch.cuda.synchronize()
    launches_per_step = int(lib.vlfm_launch_count() - n0)
    itm.engine.use_graph = True
    for i in range(Wm):
        step_device(i)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(K):
        cos = step_device(Wm + i)
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if args.dump_outputs and rank == 0:         # before the legs below reuse the engines' buffers
        dump_outputs(args.dump_outputs, cos, eng)
    from vlfm_b200.utils.dist import aggregate_throughput, gather_metrics, max_over_ranks

    ms_local = ms
    ms = max_over_ranks(ms, dev)                       # slowest rank defines the job
    value = aggregate_throughput(world, B, K, ms)
    # Everything below (end-to-end legs, roofline replay, CPU baseline, extra workloads) decorates the line; none of it may cost the
    # headline.  A watchdog thread prints the line with what has been measured so far and ends the process if the rest has not
    # finished inside its budget (a stuck device or subprocess call cannot be interrupted from Python).
    e2e = e2e_pageable = e2e_blocks = roof = cpu = clocks = extra = None
    per_rank = [[rank, ms_local, None]]
    def emit(extra):
        if rank != 0:
            return
        line = {
            "metric": "value-map steps/sec (ITM+cone-fuse)", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": K, "warmup": Wm, "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f16", "data": "synthetic",
            "config": {"workload": WORKLOAD if B == 1 else WORKLOAD.replace("batch=1 env/GPU", f"batch={B} env/GPU"),
                       "envs_per_gpu": B, "l2": "per-step working set 2.0 GB of weights > 126 MB L2 (no flush needed)",
                       "timing": "CUDA events, max over ranks"},
            "e2e": None if e2e is None else {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": H * W * 3 + H * W * 4 + 17 * 8,
                    "d2h_bytes_per_step": 4, "api": "BLIP2ITM.cosine + ValueMap.update_map (page-locked host numpy frames in, DMA to HBM, float out)",
                    "blocks_s": e2e_blocks, "blocks_note": "three K-step blocks, median reported",
                    "pageable_value": e2e_pageable,
                    "pageable_note": "same loop with ordinary (pageable) numpy frames: staged through the classes' page-locked buffers"},
            "gpu_launches": launches_per_step * K,
            "roofline": roof, "cpu_baseline": cpu, "clocks": clocks,
            "per_rank": [{"rank": int(r[0]), "ms": r[1], "conf_checksum": r[2]} for r in per_rank],
            "extra": extra,
        }
        print(json.dumps(line), flush=True)

    import faulthandler

    def give_up():
        faulthandler.dump_traceback(file=sys.stderr)
        try:
            if sampler.proc is not None:
                sampler.proc.terminate()
        except Exception:
            pass
        emit({"error": f"the legs after the headline did not finish within {args.extra_budget + 150:.0f} s; line printed by the watchdog (traceback on stderr)"})
        os._exit(0)

    dog = threading.Timer(args.extra_budget + 150.0, give_up)
    dog.daemon = True
    dog.start()

    # ---- e2e: public class API, host buffers, H2D/D2H inside the timed region
    vm = ValueMap(1, size=G, use_max_confidence=False, device=dev)
    itm1 = itm if B == 1 else BLIP2ITM(state_dict=sd, dims=dims, max_batch=1, device=dev)
    fr0 = frames_per_env[0]
    # the step's inputs wait in page-locked host memory (as a camera driver / simulator bridge would leave them)
    for f in fr0:
        f.rgb = torch.from_numpy(f.rgb).pin_memory().numpy()
        f.depth = torch.from_numpy(np.ascontiguousarray(f.depth, dtype=np.float32)).pin_memory().numpy()

    def step_host(i):
        f = fr0[i % NFRAMES]
        c = itm1.cosine(f.rgb, PROMPT)
        vm.update_map(np.array([c]), f.depth, f.tf, MIN_D, MAX_D, FOV)

    for i in range(Wm):
        step_host(i)
    # K steps per block, three blocks back to back, the MEDIAN block is reported (a 20-step block is ~65 ms of wall clock: one
    # scheduler hiccup on the host moves it by 10 %); all three are in the JSON line
    e2e_blocks = []
    for blk in range(3):
        barrier()
        t0 = time.perf_counter()
        for i in range(K):
            step_host(Wm + blk * K + i)
        torch.cuda.synchronize()
        e2e_blocks.append(max_over_ranks(time.perf_counter() - t0, dev))
    t_e2e = sorted(e2e_blocks)[1]
    e2e = world * K / t_e2e
    # the same loop with ORDINARY (pageable) numpy frames, as the reference's callers hand them over: staged through the
    # classes' own page-locked buffers
    fr_pg = [(np.array(f.rgb, copy=True), np.array(f.depth, copy=True), f.tf) for f in fr0]

    def step_pageable(i):
        rgb_, depth_, tf_ = fr_pg[i % NFRAMES]
        c = itm1.cosine(rgb_, PROMPT)
        vm.update_map(np.array([c]), depth_, tf_, MIN_D, MAX_D, FOV)

    for i in range(Wm):
        step_pageable(i)
    barrier()
    t0 = time.perf_counter()
    for i in range(K):
        step_pageable(Wm + i)
    torch.cuda.synchronize()
    t_pg = max_over_ranks(time.perf_counter() - t0, dev)
    e2e_pageable = world * K / t_pg
    # optional NCCL all-gather of a small per-rank metrics vector (never on the step path)
    per_rank = gather_metrics([rank, ms_local, float(eng.conf.sum().item())], dev)
    clocks = sampler.stop() if rank == 0 else None

    # ---- roofline of the dominant kernel (tcgen05 GEMM): GEMM-only replay, CUDA events
    roof = gemm_roofline(itm.engine, B, dims)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        sps, n, threads = cpu_reference(4, 1, 30.0, fr0, sd, dims)
        cpu = {"value": sps, "unit": "env-steps/s", "cores": threads, "kind": "port", "host_cpus": os.cpu_count(),
               "sample": f"{n} env-steps (fp32 HF BLIP-2 ITC forward + numpy/cv2 value-map oracle), 1 warm-up"}
    if not args.no_extra and (world == 1 or args.extra_multi):
        extra = run_extras(args, dev, world, rank, local)
    elif not args.no_extra:
        extra = {"skipped": "the extra workloads run at N=1 by default (--extra-multi runs them on every rank; profiles/r02_bench_n2.json)"}
    dog.cancel()
    emit(extra)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, cos, eng):
    """What the timed path handed its caller after the last timed step, as .npy files: the ITC cosine of every environment
    (cosine.npy, [B]) and the confidence / value grids (confidence.npy [n,G,G], value.npy [n,G,G,1], float32 as kept in HBM) of
    the first n environments, n as large as keeps the files under 64 MB (all of them up to 7 envs at G=1000)."""
    os.makedirs(out_dir, exist_ok=True)
    cosine = cos.float().cpu().numpy()
    per_env = (eng.conf[0].numel() + eng.value[0].numel()) * 4
    n = max(1, min(eng.batch, (DUMP_BYTES - cosine.nbytes - 4096) // per_env))
    np.save(os.path.join(out_dir, "cosine.npy"), cosine)
    np.save(os.path.join(out_dir, "confidence.npy"), eng.conf[:n].cpu().numpy())
    np.save(os.path.join(out_dir, "value.npy"), eng.value[:n].cpu().numpy())


EXTRAS_MARK = "VLFM_EXTRAS_JSON "


def extras_names(EB):
    return ["configs1_b%d" % EB, "configs2_full_step", "configs3_slice", "configs4_slice"]


def run_extras(args, dev, world, rank, local):
    """The extra workloads run in a CHILD process (`bench.py --extras-child`, same GPU) under a hard time limit: whatever happens
    in there -- an exception, a stuck device call -- costs at most the `extra` block, never the line.  The parent only aggregates:
    `value` of each entry = whole-job env-steps/s from the max over ranks of the elapsed seconds."""
    from vlfm_b200.utils.dist import max_over_ranks

    out, pending = {}, []
    try:
        env = dict(os.environ)
        env["LOCAL_RANK"], env["RANK"] = str(local), str(rank)
        cmd = [sys.executable, os.path.abspath(__file__), "--extras-child", "--extra-batch", str(args.extra_batch)]
        def last_result(stdout):
            if isinstance(stdout, bytes):
                stdout = stdout.decode("utf-8", "replace")
            lines = [l for l in (stdout or "").splitlines() if l.startswith(EXTRAS_MARK)]
            return json.loads(lines[-1][len(EXTRAS_MARK):]) if lines else None

        try:
            r = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=args.extra_budget)
            got = last_result(r.stdout)
            if got:
                out, pending = got["out"], got["pending"]
            else:
                out = {"error": f"extras child ended with code {r.returncode} and no result: {r.stderr[-300:]}"}
        except subprocess.TimeoutExpired as te:      # keep what the child had finished (it prints a cumulative line per workload)
            got = last_result(te.stdout)
            if got:
                out, pending = got["out"], got["pending"]
            out["error"] = f"extras child exceeded {args.extra_budget:.0f} s and was killed; entries above are the workloads it had finished"
    except Exception as e:
        out = {"error": repr(e)}
    for nme in extras_names(args.extra_batch):          # the same four collectives on every rank, whatever happened locally
        ent = out.get(nme) if isinstance(out.get(nme), dict) else None
        idx = ent.get("value") if ent else None
        ok = ent is not None and isinstance(idx, int) and "error" not in ent and idx < len(pending)
        worst = max_over_ranks(pending[idx][2] if ok else 1e30, dev)
        if ent is not None and "error" not in ent:
            if worst >= 1e29 or not ok:
                ent["error"] = "failed on another rank"; ent["value"] = None
            else:
                envs, steps, _ = pending[idx]
                ent["value"] = world * envs * steps / worst
    return out


def extras_child(args):
    import torch

    from vlfm_b200.vlm.blip2_config import Blip2Dims, random_state_dict

    local, rank = int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    dims = Blip2Dims()
    def progress(out, pending):          # a cumulative result line after every workload: a later stall costs only what follows
        print(EXTRAS_MARK + json.dumps({"out": out, "pending": pending}), flush=True)

    out, pending = extras_local(args, dev, rank, random_state_dict(dims, 0), dims, progress)
    progress(out, pending)


def extras_local(args, dev, rank, sd, dims, progress=lambda out, pending: None):
    """The other BASELINE.json configs, a few steps each, on this rank's GPU (env shards, no collective): configs[1] at 32 env/GPU,
    configs[2] (full step, 32 envs), a configs[3] slice (32 env/GPU, 2000^2 grid) and a configs[4] slice (1024^2 RGB-D,
    4000^2 x 0.025 m grid, 8 env/GPU).  Returns (entries, [(envs, steps, seconds)]): an entry's `value` is an index into the list."""
    import torch

    from vlfm_b200.mapping.value_map import ValueMapBatch
    from vlfm_b200.utils.full_step import FullStep, grid_bytes
    from vlfm_b200.vlm.blip2itm import BLIP2ITM
    from vlfm_b200.vlm.grounding_dino import GroundingDINO

    pk, src = peaks()
    hbm = float(pk["hbm_gbs"])
    out = {"peak_hbm_gbs": hbm, "peak_source": src}
    EB = args.extra_batch
    itm = BLIP2ITM(state_dict=sd, dims=dims, max_batch=EB, device=dev)

    # every rank records its own elapsed seconds; ONE max-over-ranks at the end turns them into whole-job values (an extra
    # that fails on one rank must not desynchronise the collective)
    pending = []

    def agg(envs, steps, seconds):
        pending.append((envs, steps, seconds))
        return len(pending) - 1

    # ---- configs[1] at EB env/GPU: ITC + cone-fuse, inputs resident in HBM
    try:
        eng = ValueMapBatch(EB, 1, size=G, use_max_confidence=False, device=dev)
        from vlfm_b200.utils.synthetic import trajectory

        nfr = 4
        fr = [trajectory(1000 + rank * EB + e, nfr, h=H, w=W, with_rgb=True, bound_m=15.0) for e in range(EB)]
        rgb = torch.from_numpy(np.stack([np.stack([f[i].rgb for f in fr]) for i in range(nfr)])).to(dev)
        depth = torch.from_numpy(np.stack([np.stack([f[i].depth for f in fr]) for i in range(nfr)])).to(dev)
        tfs = torch.from_numpy(np.stack([np.stack([f[i].tf for f in fr]) for i in range(nfr)])).to(dev)

        def st(i):
            j = i % nfr
            cos = itm.cosine_device(rgb[j], PROMPT)
            eng.update(cos.double().view(EB, 1), depth[j], tfs[j], MIN_D, MAX_D, FOV)

        for i in range(3):
            st(i)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        n = 6
        e0.record()
        for i in range(n):
            st(3 + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        roof = gemm_roofline(itm.engine, EB, dims)
        out["configs1_b%d" % EB] = {"workload": WORKLOAD.replace("batch=1 env/GPU", f"batch={EB} env/GPU"), "value": agg(EB, n, ms * 1e-3),
                                    "unit": "env-steps/s", "ms_per_step": ms / n, "steps": n, "gemm_roofline": {k: roof[k] for k in ("achieved", "peak", "frac", "unit", "launches_per_step", "gemm_ms_per_step")}}
        del eng, rgb, depth, tfs, fr
    except Exception as e:   # an extra never takes the headline down with it
        out["configs1_b%d" % EB] = {"error": repr(e)}
    torch.cuda.empty_cache()
    progress(out, pending)

    gd = None
    try:
        gd = GroundingDINO(device=dev, synthetic=True)
    except Exception as e:
        out["gdino_error"] = repr(e)

    def full(name, workload, B, h, w, g, ppm, steps, warm, bound, release=True):
        # warm >= 3: the map update is captured into a CUDA graph on its third call with the same buffers (ObstacleMapBatch.update)
        try:
            fs = FullStep(dev, B, h, w, g, ppm, itm, gd, frames_per_env=steps + warm, seed0=2000 + rank * B, bound_m=bound)
            r = fs.run(steps, warm)
            roofs = fs.grid_rooflines(hbm)
            out[name] = {"workload": workload, "value": agg(B, steps, r["wall_s"]), "unit": "env-steps/s", "ms_per_step": r["ms_per_step"],
                         "steps": steps, "warmup": warm, "envs_per_gpu": B, "component_ms_per_step": r["component_ms_per_step"], "component_note": r.get("component_note"),
                         "frontiers_per_env_step": r["frontiers_per_env_step"], "grid_bytes_per_env_step": r["grid_bytes_per_env_step"],
                         "grid_rooflines": roofs,
                         "timing": "host wall clock around whole steps (H2D of the page-locked RGB-D batch and D2H of the frontier lists inside), max over ranks; components by CUDA events"}
            del fs
        except Exception as e:
            out[name] = {"workload": workload, "error": repr(e)}
        if release:        # hand the cached blocks back only when the next workload has different shapes: re-growing the detector's
            torch.cuda.empty_cache()   # temporaries costs cudaMalloc calls inside the next workload's first steps
        progress(out, pending)

    full("configs2_full_step", f"configs[2]: full step (GroundingDINO + BLIP-2 ITC + Obstacle/Value/Frontier update), batch={EB} envs/GPU, 640x480 RGB-D, 1000^2 grid",
         EB, H, W, 1000, 20, 4, 3, 15.0, release=False)
    full("configs3_slice", f"configs[3] slice: full step, {EB} envs/GPU (256 envs = 32/GPU x 8), 640x480 RGB-D, 2000^2 x 0.05 m grid",
         EB, H, W, 2000, 20, 4, 4, 30.0)
    b4 = max(1, EB // 4)
    full("configs4_slice", f"configs[4] slice: full step, {b4} envs/GPU (64 envs on 8 GPUs), 1024x1024 RGB-D, ViT-g at 224 (reference semantics), 4000^2 x 0.025 m grid",
         b4, 1024, 1024, 4000, 40, 4, 4, 30.0)
    return out, pending


def gemm_roofline(engine, B, dims):
    """Replay only the forward's GEMM launches (same shapes/buffers) and time them with CUDA events."""
    import torch

    from vlfm_b200 import _lib

    pk, src = peaks()
    calls = []
    orig, orig_x2 = engine._gemm, engine._gemm_x2

    def rec(a, w, bias, epi, out):
        calls.append((orig, (a, w, bias, epi, out), a, w))
        orig(a, w, bias, epi, out)

    def rec_x2(a, al, w, wl, bias, epi, out, out_lo=None):       # the Q-Former's float32-grade GEMMs (algorithmic FLOPs: 2MNK)
        calls.append((orig_x2, (a, al, w, wl, bias, epi, out, out_lo), a, w))
        orig_x2(a, al, w, wl, bias, epi, out, out_lo)

    # the replay times the GEMM launches alone: residual GEMMs are replayed with the plain residual epilogue (same tiles and
    # split-K plan as the step's partial-sum epilogue; the reduce/LayerNorm launches are not GEMMs and are not replayed)
    orig_fuse = engine.fuse_ln
    engine.fuse_ln = False
    engine._gemm, engine._gemm_x2 = rec, rec_x2
    mid = torch.empty(B, H, dims.image, 3, dtype=torch.uint8, device=engine.dev)
    img = torch.zeros(B, H, W, 3, dtype=torch.uint8, device=engine.dev)
    engine._forward_impl(img, mid)
    engine._gemm, engine._gemm_x2 = orig, orig_x2
    engine.fuse_ln = orig_fuse
    torch.cuda.synchronize()
    # dominant kernel = the fp16 tcgen05 GEMM (the ViT: 97.5 % of the FLOPs).  The Q-Former's x2 launches are a different kernel
    # (three MMAs per product, float32-grade) and their residual GEMMs only split K together with the partial-sum LayerNorm launch:
    # they are counted, not replayed.
    x2_calls = [c for c in calls if c[0] is orig_x2]
    calls = [c for c in calls if c[0] is orig]
    flops = sum(2.0 * a.shape[0] * w.shape[0] * a.shape[1] for _, _, a, w in calls)
    x2_flops = sum(2.0 * a.shape[0] * w.shape[0] * a.shape[1] for _, _, a, w in x2_calls)
    for _ in range(2):
        for fn, c, _, _ in calls:
            fn(*c)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 5
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        for fn, c, _, _ in calls:
            fn(*c)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    ach = flops / (ms * 1e-3) / 1e12
    peak = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
    traffic = None
    if B == 1:  # dram__bytes_read+write per launch from the committed ncu capture of this same workload
        try:
            with open(os.path.join(ROOT, "profiles", "r01_gemm_traffic_b1.json")) as fh:
                traffic = json.load(fh)["dram_bytes_per_launch"]
        except Exception:
            traffic = None
    return {"kernel": "gemm_f16_tcgen05_kernel (1-CTA 128xBN tiles at batch 1; 2-CTA persistent 256x256 tiles for large M)", "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s",
            "frac": ach / peak, "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram__bytes_read.sum+dram__bytes_write.sum, profiles/r01_gemm_traffic_b1.json)",
            "algorithmic_bytes_per_launch": sum(2.0 * (w.numel() + a.numel()) for fn, _, a, w in calls) / len(calls), "peak_source": f"{src} (sustained dense bf16)",
            "launches_per_step": len(calls), "flops_per_launch_avg": flops / len(calls),
            "not_replayed": {"kernel": "gemm_f16x2_tcgen05_kernel (Q-Former, float32-grade)", "launches_per_step": len(x2_calls),
                             "share_of_gemm_flops": x2_flops / max(flops + x2_flops, 1.0)},
            "us_per_launch_avg": ms * 1e3 / len(calls), "gemm_ms_per_step": ms}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=1, help="environments per GPU")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--extra-budget", type=float, default=240.0, help="seconds the extra workloads (a child process) may take before they are killed and the line is printed without them")
    ap.add_argument("--no-extra", action="store_true", help="skip the configs[1]@32 / [2] / [3] / [4] slices")
    ap.add_argument("--extra-batch", type=int, default=32, help="envs per GPU of the extra slices")
    ap.add_argument("--extra-multi", action="store_true", help="run the extra workloads on every rank of a multi-GPU launch too")
    ap.add_argument("--extras-child", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the cosines and value-map grids of the last timed step as DIR/<name>.npy (rank 0's environments); "
                         "the inputs are seeded, so two builds run with the same arguments can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs records the b200 path")
    if args.extras_child:
        extras_child(args)
    elif args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
