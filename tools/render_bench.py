"""Cost of batched rendering next to the solver step (profiles/r03_render_bench.json).

For CylinderJet2D-easy at B = 256 and Airfoil2D-easy at B = 64, in steady state: CUDA-event times of ``env.step`` alone and of
``env.step`` + ``env.render()``, alternated pair by pair in one process; then, in a run of their own under torch.profiler, the
device times of the two render kernels, with the bytes each must move (from the shapes) over its time against the 7.7 TB/s
HBM3e bandwidth of one B200.  Card name and power limit are read in the same run.

    python tools/render_bench.py [--pairs 20] [--out profiles/r03_render_bench.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

PEAK_BYTES_PER_S = 7.7e12
CASES = [("CylinderJet2D-easy-v0", 256), ("Airfoil2D-easy-v0", 64)]


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True)
        name, power, clock = (s.strip() for s in out.splitlines()[0].split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:                                           # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def kernel_bytes(env, B):
    """bytes the two kernels must move for one render() of the default field: the map once, every cell value of the field's
    channels once, the image written (gather) / read + the RGB written (colour)"""
    (rowptr, col, w), (H, W) = env._render_map(None)
    src, _ = env._render_source(None)
    P = H * W
    gather = (rowptr.numel() + col.numel()) * 4 + w.numel() * 4 + B * src.shape[1] * src.shape[2] * 4 + B * P * 4 + B * 8
    colour = B * P * 4 + B * P * 3 + B * 8 + 768
    return dict(gather=gather, colour=colour, pixels=P, nnz=int(col.numel()))


def bench(env_id, B, pairs):
    import fluidgym_b200 as fg
    env = fg.make(env_id, n_envs=B)
    env.reset(seed=0)
    a = torch.zeros(env._zero_action.shape, device=env.device)
    for _ in range(3):                                               # warm-up of both variants (map build, module load)
        env.step(a)
        env.render()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    t_step, t_both, t_render = [], [], []
    for i in range(pairs):
        if env._n_steps + 2 >= env.episode_length:
            env.reset(seed=i)
        for with_render, acc in ((False, t_step), (True, t_both)):
            ev[0].record()
            env.step(a)
            if with_render:
                env.render()
            ev[1].record()
            ev[1].synchronize()
            acc.append(ev[0].elapsed_time(ev[1]))
    for _ in range(pairs):
        ev[0].record()
        env.render()
        ev[1].record()
        ev[1].synchronize()
        t_render.append(ev[0].elapsed_time(ev[1]))
    step, both = statistics.median(t_step), statistics.median(t_both)
    res = dict(env=env_id, B=B, pairs=pairs, step_ms=step, step_plus_render_ms=both, render_alone_ms=statistics.median(t_render),
               render_overhead_pct=100.0 * (both - step) / step, step_ms_all=t_step, step_plus_render_ms_all=t_both,
               env_steps_per_s=B / (step / 1e3))
    # kernel times in a run of their own
    from torch.profiler import ProfilerActivity, profile
    n = 20
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            env.render()
        torch.cuda.synchronize()
    by = kernel_bytes(env, B)
    for ka in prof.key_averages():
        for kname, key in (("k_render_gather", "gather"), ("k_render_colour", "colour")):
            if kname in ka.key:
                t = ka.device_time_total / ka.count * 1e-6             # us -> s
                res[f"{kname}_us"] = t * 1e6
                res[f"{kname}_bytes"] = by[key]
                res[f"{kname}_GBps"] = by[key] / t / 1e9
                res[f"{kname}_share_of_7.7TBps"] = by[key] / t / PEAK_BYTES_PER_S
    res.update(pixels=by["pixels"], nnz=by["nnz"])
    del env
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_render_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("render_bench needs a GPU")
    out = dict(card=card(), cases=[bench(e, B, args.pairs) for e, B in CASES])
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    for c in out["cases"]:
        print(json.dumps({k: v for k, v in c.items() if not k.endswith("_all")}))


if __name__ == "__main__":
    main()
