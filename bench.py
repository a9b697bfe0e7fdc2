#!/usr/bin/env python
"""Benchmark of the fluid-solver step (BASELINE.json: env-steps/sec = PISO solver steps x envs per second).

    python bench.py --gpus N --steps K --warmup W            # this repo (hand-written sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K ...  # the unmodified reference on the same box
    python bench.py ... --dump-outputs DIR                   # + what the last timed env.step() returned, as DIR/<name>.npy

One bench "step" = one RL ``env.step()`` of the whole batch = 25 solver (PISO) steps per environment incl.
jet actuation, advective outflow update, drag/lift integration and sensor sampling.
Workload (BASELINE.json configs[1]): CylinderJet2D-easy-v0 (5-block O-grid, 14 232 cells, fp32), 256
environments per GPU, synthetic initial state = projected initial field + per-environment Gaussian noise,
random jet actions.  Environments are independent -> weak scaling over GPUs with no collective on the
data path (SURVEY.md section 8e).
"""
from __future__ import annotations

import argparse
import contextlib
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

if os.environ.get("FGB_REF_CHILD_SHIMS") == "1" and __name__ != "__main__":
    # a worker process of the reference's own ParallelFluidEnv (envs/parallel_env.py:162-175, start method "spawn") imports the
    # parent's main module before it unpickles its target: make the unmodified reference importable there as well
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_shims as _ref_shims
    _ref_shims.install()

ENV_ID = "CylinderJet2D-easy-v0"
METRIC = "env-steps/sec (solver steps x envs)"
UNIT = "env-steps/s"
CG_BYTES_PER_CELL_ITER = 64      # SURVEY.md section 8(d): K_cg = S + 11 floats = 64 B per cell and iteration in 2-D
BICG_BYTES_PER_CELL_ITER = 248   # K_bicg = D (2S + 21) floats


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi sampling during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.f = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.gpu)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        try:
            self.proc.terminate()
            self.proc.wait(timeout=5)
            self.f.close()
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = [float(r[1]) for r in rows]
            reasons = set()
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            for r in rows:
                for k, nme in enumerate(names):
                    if len(r) > 5 + k and r[5 + k].strip().lower() == "active":
                        reasons.add(nme)
            if sm:
                out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(rows[0][2]), "reasons": sorted(reasons),
                       "samples": len(sm), "power_w_max": max(float(r[3]) for r in rows)}
        except Exception as e:  # pragma: no cover
            out["error"] = str(e)
        finally:
            try:
                os.unlink(self.path)
            except Exception:
                pass
        return out


def dist_setup(n_gpus):
    import torch
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    return rank, world, local


def barrier(world):
    import torch
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


def max_over_ranks(x, world, device):
    import torch
    if world == 1:
        return float(x)
    import torch.distributed as dist
    t = torch.tensor([float(x)], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(x, world, device):
    import torch
    if world == 1:
        return float(x)
    import torch.distributed as dist
    t = torch.tensor([float(x)], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


# ------------------------------------------------------------------------------------------------
def cpu_baseline(env, n_sim_steps=12):
    """CPU restatement (oracle/piso_oracle.c) timed on the host cores, one environment per thread (the batch is embarrassingly
    parallel; ctypes releases the GIL), starting from the states of the first environments after the GPU warm-up: a bounded
    sample of the same workload."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from concurrent.futures import ThreadPoolExecutor
    from oracle import Oracle
    cd = env.cd
    s = env.solver
    cores = max(1, min(os.cpu_count() or 1, env.n_envs))
    out_mask = env.solver._tab["b_out"].cpu().numpy().astype(np.uint8)
    jobs = []
    for e in range(cores):
        jobs.append((Oracle(cd.sizes, cd.btype, cd.bconn, cd.T, cd.bT, s.bvel[e].cpu().numpy(), float(cd.visc)),
                     s.u[e].cpu().numpy().copy(), s.p[e].cpu().numpy().copy()))

    def run(job):
        orc, u, p = job
        n = 0
        for _ in range(n_sim_steps):
            k, _, _ = orc.sim_step(u, p, env.dt, env.cfl, out_mask=out_mask, adj=cd.b_cell, char_vel=[1.0, 0.0])
            n += k
        return n

    t0 = time.perf_counter()
    with ThreadPoolExecutor(cores) as ex:
        nsub = sum(ex.map(run, jobs))
    el = time.perf_counter() - t0
    return {"value": nsub / el, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{n_sim_steps} solver steps of {cores} environments (grid / states of the first environments after warm-up), "
                      f"oracle/piso_oracle.c, one environment per host thread, {os.cpu_count()} host cores present"}


def _snapshot(env):
    """Solver + actuator state, so that the device-resident and the end-to-end loops time the SAME physical work
    (iteration counts, and with them the cost of a step, drift as the flow develops)."""
    s = env.solver
    snap = {"u": s.u.clone(), "p": s.p.clone(), "bvel": s.bvel.clone(), "ures": s.buffer("ures").clone()}
    if getattr(s, "has_scalar", False):
        snap.update(T=s.T.clone(), sbval=s.sbval.clone(), vsrc=s.vsrc.clone())
    if hasattr(env, "last_control"):
        snap["last_control"] = env.last_control.clone()
    return snap


def _restore(env, snap):
    s = env.solver
    s.u.copy_(snap["u"]); s.p.copy_(snap["p"]); s.bvel.copy_(snap["bvel"]); s.buffer("ures").copy_(snap["ures"])
    if "T" in snap:
        s.T.copy_(snap["T"]); s.sbval.copy_(snap["sbval"]); s.vsrc.copy_(snap["vsrc"])
    if "last_control" in snap:
        env.last_control.copy_(snap["last_control"])
    env._n_steps = 0


DUMP_BYTES = 64 << 20


def _step_arrays(result):
    """The arrays a caller receives from one env.step() -- observation, reward, terminated, truncated, info -- flattened to
    host float arrays (float64 where float32 would round: double, integer and boolean values)."""
    import torch
    obs, reward, terminated, truncated, info = result
    named = {"reward": reward, "terminated": terminated, "truncated": truncated}
    named.update({f"obs_{k}": v for k, v in obs.items()} if isinstance(obs, dict) else {"obs": obs})
    named.update({f"info_{k}": v for k, v in info.items()})
    out = {}
    for name, v in named.items():
        a = v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)
        out[name] = a.astype(np.float32 if a.dtype in (np.float16, np.float32) else np.float64)
    return out


def dump_outputs(arrays, path, tag=""):
    """Writes ``path/<name><tag>.npy``.  Arrays are sampled at fixed, seeded flat positions where the whole set would exceed
    DUMP_BYTES, so that two builds run with the same arguments write comparable files."""
    os.makedirs(path, exist_ok=True)
    budget = DUMP_BYTES // max(len(arrays), 1)
    for name, a in sorted(arrays.items()):
        if a.nbytes > budget:
            keep = np.sort(np.random.default_rng(0).choice(a.size, budget // a.itemsize, replace=False))
            a = a.reshape(-1)[keep]
        np.save(os.path.join(path, f"{name}{tag}.npy"), a)


# ------------------------------------------------------------------------------------------------
def extras(args, rank, world, local, dev):
    """Short records of the other BASELINE.json configs (kept bounded; failures are reported, never fatal):
    config 3 (RBC2D multi-agent, env batch, weak), config 4 (Airfoil2D-medium differentiable rollout, N = 1 only),
    config 5 (TCFLarge, one environment: plain solver at N = 1, z-slab decomposition over the N GPUs otherwise)."""
    import torch
    import fluidgym_b200
    out = {}
    # ---- config 3 ----
    try:
        B = args.extra_rbc_envs
        env = fluidgym_b200.make("RBC2D-easy-v0", n_envs=B, device=str(dev), use_marl=True)
        env.reset(seed=42 + rank)
        env.episode_length = 10 ** 9
        g = torch.Generator(device=dev).manual_seed(5 + rank)
        acts = torch.rand(6, *env._zero_action.shape, device=dev, generator=g) * 2 - 1
        for i in range(3):
            env.step(acts[i])
        barrier(world)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        nsub = 0
        for i in range(3):
            env.step(acts[3 + i])
            nsub += env.last_substeps
        e1.record()
        barrier(world)
        ms = max_over_ranks(e0.elapsed_time(e1), world, dev)
        out["rbc2d_marl"] = {"workload": f"RBC2D-easy-v0 use_marl x{B} envs per GPU (configs[2]), 3 env.step()", "n_gpus": world,
                             "value": sum_over_ranks(B * nsub, world, dev) / (ms / 1e3), "unit": UNIT, "ms_per_step": ms / 3, "scaling": "weak"}
        del env
        torch.cuda.empty_cache()
    except Exception as e:
        out["rbc2d_marl"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    # ---- config 4 ----
    if world == 1:
        try:
            n_env_steps = args.extra_airfoil_steps
            env = fluidgym_b200.make("Airfoil2D-medium-v0", n_envs=1, device=str(dev), differentiable=True)
            env.reset(seed=42)
            torch.cuda.reset_peak_memory_stats()
            a = (torch.linspace(-1, 1, 3, device=dev).repeat(1, 1) * 0.5).requires_grad_(True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            total, nsub = 0.0, 0
            for _ in range(n_env_steps):
                obs, r, *_ = env.step(a)
                total = total + r.sum()
                nsub += env.last_substeps
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            total.backward()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            env.detach()
            out["airfoil2d_diff"] = {"workload": f"Airfoil2D-medium-v0 differentiable, {n_env_steps} env.step() = {n_env_steps * env.n_sim_steps} "
                                                 f"solver steps ({nsub} substeps) forward + backward (configs[3])",
                                     "forward_s": t1 - t0, "backward_s": t2 - t1, "backward_over_forward": (t2 - t1) / (t1 - t0),
                                     "peak_mem_GB": torch.cuda.max_memory_allocated() / 2 ** 30,
                                     "grad_action": [float(x) for x in a.grad.flatten()]}
            del env
            torch.cuda.empty_cache()
        except Exception as e:
            out["airfoil2d_diff"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    # ---- config 5 ----
    try:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import tcf_slab_bench
        rec = tcf_slab_bench.run(large=True, steps=args.extra_tcf_steps, warmup=3, plain=(world == 1), rank=rank, world=world, local=local)
        rec["scaling"] = "strong"
        rec["note"] = ("one TCFLarge environment; identical work at every N (same state, same steps): compare ms_per_substep, "
                       "cg / bicg iterations and checksum_u2 across the N = 1 (plain solver) / 2 / 4 / 8 lines")
        out["tcf_large"] = rec
    except Exception as e:
        out["tcf_large"] = {"error": f"{type(e).__name__}: {e}"[:300]}
    return out


def run_ours(args):
    import torch
    import fluidgym_b200
    from fluidgym_b200 import native

    rank, world, local = dist_setup(args.gpus)
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    B = args.envs
    env_id = ENV_ID if args.workload == "cylinder" else "RBC2D-easy-v0"
    kw = {} if args.workload == "cylinder" else {"use_marl": True}
    if args.cg_impl is not None:
        kw["cg_impl"] = args.cg_impl
    env = fluidgym_b200.make(env_id, n_envs=B, device=str(dev), **kw)
    args.cg_impl = int(env.solver.options.cg_impl)
    N = env.cd.N
    env.reset(seed=42 + rank)
    gen = torch.Generator(device=dev).manual_seed(1000 + rank)
    env.solver.u += 0.025 * torch.randn(env.solver.u.shape, device=dev, generator=gen)
    env.solver.p += 0.025 * torch.randn(env.solver.p.shape, device=dev, generator=gen)
    cpu_gen = torch.Generator().manual_seed(7 + rank)
    total = args.warmup + 2 * args.steps
    actions_host = (torch.rand(total, *env._zero_action.shape, generator=cpu_gen) * 2 - 1).pin_memory()
    actions_dev = actions_host.to(dev)
    env.episode_length = 10 ** 9

    for i in range(args.warmup):
        env.step(actions_dev[i])
    torch.cuda.synchronize()
    lib, h = env.lib, env.solver.handle
    snap = _snapshot(env)

    # ---- kernel-resident timing: inputs already in HBM ------------------------------------------
    it0 = env.solver.buffer("iter_total").view(torch.int64).clone()
    l0 = lib.fgb_launch_count(h)
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    barrier(world)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    nsub = 0
    for i in range(args.steps):
        last = env.step(actions_dev[args.warmup + i])
        nsub += env.last_substeps
    e1.record()
    barrier(world)
    ms_local = e0.elapsed_time(e1)
    clk = clocks.stop() if rank == 0 else None
    launches = lib.fgb_launch_count(h) - l0
    it1 = env.solver.buffer("iter_total").view(torch.int64).clone()
    d_it = (it1 - it0).cpu().numpy().reshape(B, 2)
    ms = max_over_ranks(ms_local, world, dev)
    env_substeps = sum_over_ranks(B * nsub, world, dev)
    value = env_substeps / (ms / 1e3)
    if args.dump_outputs:
        dump_outputs(_step_arrays(last), args.dump_outputs, "" if world == 1 else f".rank{rank}")

    # ---- per-kernel durations for the roofline block: the same steps once more with ONE environment group, so that every
    #      launch runs alone on the GPU and its CUDA-event duration is the kernel's own (in the timed region above the
    #      groups' kernels overlap on purpose) ------------------------------------------------------------------------------
    _restore(env, snap)
    n_groups = env.solver.groups
    env.solver.set_groups(1)
    native.check(lib.fgb_profile_enable(h, 1), "profile_enable")
    itp0 = env.solver.buffer("iter_total").view(torch.int64).clone()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record()
    n_prof = min(args.steps, 2)
    for i in range(n_prof):
        env.step(actions_dev[args.warmup + i])
    p1.record()
    torch.cuda.synchronize()
    ms_serial = p0.elapsed_time(p1)
    ms_prof = (C.c_double * 4)()
    cnt_prof = (C.c_int64 * 4)()
    native.check(lib.fgb_profile_read(h, ms_prof, cnt_prof, 1), "profile_read")
    native.check(lib.fgb_profile_enable(h, 0), "profile_enable")
    d_itp = (env.solver.buffer("iter_total").view(torch.int64) - itp0).cpu().numpy().reshape(B, 2)
    env.solver.set_groups(n_groups)

    # ---- end-to-end through the public API with host buffers --------------------------------------
    obs_probe, rew_probe, _, _, _ = env.step(actions_dev[args.warmup])
    _restore(env, snap)                 # same state and the same actions as the device-resident loop above
    torch.cuda.synchronize()
    obs_host = {k2: torch.empty(v.shape).pin_memory() for k2, v in obs_probe.items()}
    rew_host = torch.empty(rew_probe.shape).pin_memory()
    barrier(world)
    t0 = torch.cuda.Event(enable_timing=True)
    t1 = torch.cuda.Event(enable_timing=True)
    t0.record()
    nsub_e = 0
    for i in range(args.steps):
        a = actions_host[args.warmup + i].to(dev, non_blocking=True)
        obs, rew, _, _, info = env.step(a)
        for k2, v in obs.items():
            obs_host[k2].copy_(v, non_blocking=True)
        rew_host.copy_(rew, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        nsub_e += env.last_substeps
    t1.record()
    barrier(world)
    ms_e = max_over_ranks(t0.elapsed_time(t1), world, dev)
    e2e_value = sum_over_ranks(B * nsub_e, world, dev) / (ms_e / 1e3)
    h2d = actions_host[0].numel() * 4
    d2h = (sum(v.numel() for v in obs_host.values()) + rew_host.numel()) * 4

    # ---- roofline of the dominant kernel (pressure CG) ---------------------------------------------
    peak, peak_src = peaks()
    cg_ms, cg_launches = ms_prof[0], int(cnt_prof[0])
    cg_bytes = float(d_itp[:, 0].sum()) * N * CG_BYTES_PER_CELL_ITER
    achieved = cg_bytes / (cg_ms / 1e3) / 1e9 if cg_ms > 0 else 0.0
    traffic = None
    tp = os.path.join(ROOT, "profiles", "cg_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        except Exception:
            traffic = None
    roof = {"bound": "hbm", "kernel": {0: "k_cg", 1: "k_cg_cluster", 2: "k_cg_cluster", 3: "k_cg_cluster_mb", 4: "k_cg_smem", 5: "k_cg_smem", 6: "k_cg_cluster_mb<PUSH>", 7: "k_cg_cluster_mb<PUSH,256x14>", 8: "k_cg_cluster_mb<PUSH,256x7,2 CTAs/SM>", 11: "k_cg_strip<480,17>", 12: "k_cg_strip2<480,9>"}.get(args.cg_impl, f"cg_impl {args.cg_impl}"), "achieved": achieved, "peak": peak,
            "peak_source": peak_src, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
            "algorithmic_bytes_per_launch": cg_bytes / max(cg_launches, 1), "avg_launch_ms": cg_ms / max(cg_launches, 1),
            "launches": cg_launches, "share_of_step": cg_ms / ms_serial,
            "measured_on": f"{n_prof} env.step() replayed after the timed region with one environment group (kernels run alone); "
                           f"the timed region runs {n_groups} groups on concurrent streams",
            "note": "on-chip (cluster-resident) CG: algorithmic bytes are the SURVEY 8(d) streaming figure; measured DRAM "
                    "traffic is far lower because x/r/p and the stencil stay in registers/shared memory, so frac > 1 is not a bound; "
                    "`traffic` is the ncu capture of profiles/cg_traffic.json (not re-measured in this run)",
            # the ceilings that do bind this kernel, from the same ncu capture (profiles/r02_ncu_cg_strip_480x17.txt and
            # profiles/r02_cg_strip_development.md): a latency-bound dependent chain with 15 warps per SM
            "binding_ceilings": {"issue_slots_active_pct": 31.7, "shared_memory_pipe_pct": 42, "warps_per_sm": 15,
                                 "cycles_per_iteration": 7100, "warp_instructions_per_iteration": 625,
                                 "source": "ncu --set full, static (captured once per kernel change, see profiles/)"} if args.cg_impl == 11 else None}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{env_id} x{B} envs per GPU (BASELINE.json configs[{1 if args.workload == 'cylinder' else 2}]); "
                               f"step = env.step() = {env.n_sim_steps} solver steps (adaptive CFL substeps)",
                   "cells_per_env": N, "envs_per_gpu": B, "parallelism": f"env-batch x{world} (no collective)",
                   "l2_policy": f"working set {B} envs x {N * 45 * 4 / 1e6:.1f} MB > 126 MB L2 (inputs larger than L2)",
                   "cg_impl": args.cg_impl},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e / args.steps},
        "gpu_launches": int(launches),
        "roofline": roof,
        "solver": {"cg_iters_per_solve": float(d_it[:, 0].sum()) / max(B * nsub * 2, 1),
                   "bicg_iters_per_rhs": float(d_it[:, 1].sum()) / max(B * nsub * 2, 1),
                   "substeps_per_sim_step": nsub / (args.steps * env.n_sim_steps),
                   "rl_env_steps_per_s": value / (env.n_sim_steps * max(nsub / (args.steps * env.n_sim_steps), 1e-9)),
                   "time_share_ms_serial_replay": {"cg": ms_prof[0], "bicgstab": ms_prof[1], "assembly": ms_prof[2], "total": ms_serial,
                                                "env_steps": n_prof},
                   "environment_groups": n_groups},
        "clocks": clk,
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline and args.workload == "cylinder":
        line["cpu_baseline"] = cpu_baseline(env, args.cpu_steps)
    if not args.no_extras and args.workload == "cylinder":
        del env
        torch.cuda.empty_cache()
        ex = extras(args, rank, world, local, dev)
        line["extra"] = ex
    if rank == 0:
        print(json.dumps(line))
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm.  The reference has NO CPU implementation of this path (FluidEnv.reset raises without
    CUDA, envs/fluid_env.py:885-886): when the unmodified reference (baseline/_ref, built by
    oracle/build_ref.sh) and a GPU are present it is run through its own public API -- one environment in this
    process (fluidgym.make -> reset -> step; its native ops assert batch size 1) and its own batching mechanism,
    ParallelFluidEnv(cuda_ids=[gpu] * k) = k worker processes on the same GPU (envs/parallel_env.py:116-287);
    otherwise the CPU oracle port is timed.  Under torchrun every rank runs the reference on its own GPU and rank 0
    prints the sum (the per-GPU figure is in config)."""
    rank = int(os.environ.get("RANK", 0))
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    kind = args.ref_kind
    have_ref = os.path.isdir(os.path.join(ROOT, "baseline", "_ref", "fluidgym"))
    import torch
    if kind == "auto":
        kind = "cuda" if (have_ref and torch.cuda.is_available()) else "cpu"
    if kind == "cuda":
        try:
            _run_reference_cuda(args)
            return
        except Exception as e:                                   # a broken reference install must not lose the arm
            if args.ref_kind == "cuda":
                raise
            print(f"[bench] unmodified reference failed ({type(e).__name__}: {e}); timing the CPU oracle port instead",
                  file=sys.stderr)
    if rank == 0:
        _run_reference_port(args)


def _reference_actions(n, shape):
    import torch
    g = torch.Generator().manual_seed(7)
    return torch.rand(n, *shape, generator=g) * 2 - 1


def _run_reference_cuda(args):
    import torch
    import ref_shims
    ref_shims.install()
    import fluidgym
    from fluidgym.simulation.extensions import PISOtorch
    rank, world = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("gloo")
    dev = torch.device(f"cuda:{local}")
    torch.cuda.set_device(dev)
    kw = dict(load_initial_domain=False, load_domain_statistics=False, randomize_initial_state=False)

    # ---- (1) one environment in this process: timing, substep count and Krylov iterations ------------------------------
    env = fluidgym.make(ENV_ID, cuda_device=dev, **kw)
    env.reset(seed=42)
    cnt = {"n": 0, "cg": [], "bicg": []}
    orig_mat, orig_solve = PISOtorch.SetupAdvectionMatrix, PISOtorch.SolveLinear

    def counted(*a, **k):
        cnt["n"] += 1
        return orig_mat(*a, **k)

    def solve_logged(*a, **k):
        res = orig_solve(*a, **k)
        use_bicg = bool(a[6]) if len(a) > 6 else bool(k.get("useBiCG", False))
        cnt["bicg" if use_bicg else "cg"].extend(int(i.usedIterations) for i in res)
        return res

    PISOtorch.SetupAdvectionMatrix, PISOtorch.SolveLinear = counted, solve_logged
    acts = _reference_actions(args.warmup + args.steps, tuple(env._zero_action.shape))
    env._episode_length = 10 ** 9
    for i in range(args.warmup):
        env.step(acts[i].to(dev))
    torch.cuda.synchronize()
    cnt.update(n=0, cg=[], bicg=[])
    t0 = time.perf_counter()
    for i in range(args.steps):
        env.step(acts[args.warmup + i].to(dev))
    torch.cuda.synchronize()
    el1 = time.perf_counter() - t0
    nsub1 = cnt["n"]
    single = {"envs": 1, "value": nsub1 / el1, "ms_per_step": el1 / args.steps * 1e3,
              "cg_iters_per_solve": float(np.mean(cnt["cg"])) if cnt["cg"] else None,
              "bicg_iters_per_rhs": float(np.mean(cnt["bicg"])) if cnt["bicg"] else None,
              "substeps_per_env_step": nsub1 / args.steps}
    PISOtorch.SetupAdvectionMatrix, PISOtorch.SolveLinear = orig_mat, orig_solve
    del env
    torch.cuda.empty_cache()

    # ---- (2) the reference's own batching: k worker processes on this GPU, identical environments and actions ------------
    parallel = None
    k = args.ref_envs if args.ref_envs > 0 else max(1, min(8, (os.cpu_count() or 2) // 2))
    if k > 1:
        try:
            os.environ["FGB_REF_CHILD_SHIMS"] = "1"
            from fluidgym.envs.parallel_env import ParallelFluidEnv
            penv = ParallelFluidEnv(ENV_ID, cuda_ids=[local] * k, **kw)
            penv.reset(seed=42)
            pa = acts.unsqueeze(1).expand(-1, k, *acts.shape[1:]).contiguous()   # every worker replays the run above
            for i in range(args.warmup):
                penv.step(pa[i])
            t0 = time.perf_counter()
            for i in range(args.steps):
                penv.step(pa[args.warmup + i])
            elk = time.perf_counter() - t0
            parallel = {"envs": k, "value": k * nsub1 / elk, "ms_per_step": elk / args.steps * 1e3,
                        "note": "k identical environments with the actions of the single-environment run: substeps = k x its count"}
            try:
                penv.close()
            except Exception:
                pass
        except Exception as e:                                   # keep the single-environment number
            parallel = {"envs": k, "error": f"{type(e).__name__}: {e}"[:300]}
    best = single if not (parallel and "value" in parallel and parallel["value"] > single["value"]) else parallel
    value, ms = best["value"], best["ms_per_step"]
    total = value
    if world > 1:
        import torch.distributed as dist
        tt = torch.tensor([value, ms], dtype=torch.float64)
        vals = [torch.zeros_like(tt) for _ in range(world)]
        dist.all_gather(vals, tt)
        total = float(sum(v[0] for v in vals))
        ms = float(max(v[1] for v in vals))
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {"impl": "reference", "metric": METRIC, "value": total, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{ENV_ID} x{best['envs']} envs per GPU: the largest batch the reference runs on one GPU here "
                                   f"(its native ops assert batch size 1; ParallelFluidEnv = one OS process + CUDA context per "
                                   f"environment, envs/parallel_env.py:162-175); step = env.step() = 25 PISO solver steps",
                       "reference_kind": "unmodified reference CUDA extension compiled for sm_100 (baseline/_ref), its own API",
                       "per_gpu_value": value, "single_env": single, "parallel_env": parallel, "host_cores": os.cpu_count(),
                       "start_state": "reference reset (impulsive start + projection), no noise; Krylov iterations per solve are "
                                      "in single_env for comparison with the repo arm's solver block"},
            "cpu_baseline": {"value": total, "unit": UNIT, "cores": os.cpu_count(), "kind": "reference",
                             "sample": f"{args.steps} env.step() of {best['envs']} environment(s) per GPU through the reference's API; "
                                       f"the reference has no CPU solver, this is its CUDA path driven by its python loop"},
            "e2e": {"value": total, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def _run_reference_port(args):
    # CPU oracle port
    from fluidgym_b200.envs.cylinder_domain import WAKE, make_cylinder_domain
    from oracle import Oracle
    spec = make_cylinder_domain(24)
    cd = spec.prepare()
    orc = Oracle.from_compiled(cd)
    u = np.zeros((2, cd.N), np.float32)
    p = np.zeros(cd.N, np.float32)
    out = np.zeros(cd.NB, np.uint8)
    o = cd.boff[WAKE, 1]
    out[o:o + spec.blocks[WAKE].ny] = 1
    orc.update_outflow(u, out, cd.b_cell, [1.0, 0.0], 1.0, 1e-5)
    orc.make_divergence_free(u, p, 1000)
    per_step = max(1, args.cpu_steps // max(args.steps, 1))
    for _ in range(args.warmup):
        orc.sim_step(u, p, 0.01, 0.8, out_mask=out, adj=cd.b_cell, char_vel=[1.0, 0.0])
    t0 = time.perf_counter()
    nsub = 0
    for _ in range(args.steps * per_step):
        n, _, _ = orc.sim_step(u, p, 0.01, 0.8, out_mask=out, adj=cd.b_cell, char_vel=[1.0, 0.0])
        nsub += n
    el = time.perf_counter() - t0
    value = nsub / el
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{ENV_ID} x1 env, {per_step} solver steps per bench step (bounded sample)",
                       "reference_kind": "CPU oracle port (oracle/piso_oracle.c), the reference has no CPU path"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port",
                             "sample": f"{args.steps * per_step} solver steps of 1 environment"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--envs", type=int, default=256, help="environments per GPU")
    ap.add_argument("--workload", default="cylinder", choices=["cylinder", "rbc"])
    ap.add_argument("--cg-impl", type=int, default=None, help="pressure-CG implementation (default: the environment's own)")
    ap.add_argument("--ref-kind", default="auto", choices=["auto", "cuda", "cpu"])
    ap.add_argument("--ref-envs", type=int, default=0, help="worker processes of the reference's ParallelFluidEnv (0: min(8, cores / 2))")
    ap.add_argument("--cpu-steps", type=int, default=12)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the short records of BASELINE configs 3, 4, 5")
    ap.add_argument("--extra-rbc-envs", type=int, default=1024)
    ap.add_argument("--extra-airfoil-steps", type=int, default=10, help="env.step() of the differentiable airfoil rollout (5 solver steps each)")
    ap.add_argument("--extra-tcf-steps", type=int, default=10)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed env.step() returned (observation, reward, terminated, truncated, info) as "
                         "DIR/<name>.npy; under torchrun every rank writes DIR/<name>.rank<r>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    # ONE line on stdout: libraries write banners to file descriptor 1 behind python's back (NCCL prints "NCCL version ..." there when
    # the process group comes up), so fd 1 points to stderr while the run is in progress and the JSON line goes to the real stdout
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    out = os.fdopen(real_stdout, "w")
    try:
        with contextlib.redirect_stdout(out):
            if args.impl == "reference":
                run_reference(args)
            else:
                run_ours(args)
    finally:
        out.flush()


if __name__ == "__main__":
    main()
