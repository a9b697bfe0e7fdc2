"""Cost of the two substep plans of a batched differentiable rollout (profiles/r03_diff_substeps_bench.json).

CylinderJet2D-easy, B = 16, differentiable=True, one env.step (25 solver steps) from the reset state with environment b's velocity
scaled by SCALES[b], so that the environments need different numbers of substeps.  For the shared plan (the default: the most restrictive
environment sets one substep size for the batch) and the per-environment plan (``per_env_substeps=True``): substep rounds launched,
substeps summed over the environments, CUDA-event milliseconds of the forward step and of the backward pass (each ending in a device
synchronise), and the peak of allocated device memory.  The two plans alternate rep by rep in one process after one warm-up step each;
medians are reported with every sample.  Card name and power limit are read in the same run.

    python tools/diff_substeps_bench.py [--reps 5] [--out profiles/r03_diff_substeps_bench.json]
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

ENV_ID, B = "CylinderJet2D-easy-v0", 16


def card():
    try:
        out = subprocess.check_output(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], text=True)
        name, power, clock = (s.strip() for s in out.splitlines()[0].split(","))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:                                           # noqa: BLE001
        return dict(name=torch.cuda.get_device_name(0), power_limit=f"unknown ({e})")


def one_step(env, scales, action):
    """reset, diverge the states, one differentiable env.step + backward -> (forward ms, backward ms, peak bytes)"""
    env.reset(seed=0)
    with torch.no_grad():
        env.solver.u.mul_(scales[:, None, None])
    env._dstate = None
    a = action.clone().requires_grad_(True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    ev[0].record()
    _, reward, *_ = env.step(a)
    ev[1].record()
    torch.cuda.synchronize()
    ev_b = torch.cuda.Event(enable_timing=True)
    ev_b.record()
    reward.sum().backward()
    ev[2].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]), ev_b.elapsed_time(ev[2]), torch.cuda.max_memory_allocated()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_diff_substeps_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("diff_substeps_bench.py needs a CUDA device")
    import fluidgym_b200 as fg
    scales = torch.linspace(1.0, 2.5, B, device="cuda")
    action = torch.linspace(-0.5, 0.5, B, device="cuda").reshape(B, 1)
    envs = {plan: fg.make(ENV_ID, n_envs=B, differentiable=True, per_env_substeps=(plan == "per_env")) for plan in ("shared", "per_env")}
    res = {plan: dict(forward_ms=[], backward_ms=[], peak_bytes=[]) for plan in envs}
    for plan, env in envs.items():                                   # warm-up
        one_step(env, scales, action)
    for _ in range(args.reps):
        for plan, env in envs.items():
            f, b, m = one_step(env, scales, action)
            res[plan]["forward_ms"].append(f); res[plan]["backward_ms"].append(b); res[plan]["peak_bytes"].append(m)
    out = dict(card=card(), env=ENV_ID, n_envs=B, velocity_scales=[round(float(s), 4) for s in scales], reps=args.reps,
               step=dict(solver_steps=envs["shared"].n_sim_steps, dt=envs["shared"].dt, cfl=envs["shared"].cfl))
    for plan, env in envs.items():
        r = res[plan]
        per_env = env.last_substeps_per_env.cpu().tolist() if env.last_substeps_per_env is not None else None
        out[plan] = dict(rounds=env.last_substeps,
                         substeps_per_env=per_env if per_env is not None else [env.last_substeps] * B,
                         substeps_total=sum(per_env) if per_env is not None else env.last_substeps * B,
                         forward_ms=statistics.median(r["forward_ms"]), backward_ms=statistics.median(r["backward_ms"]),
                         peak_mib=max(r["peak_bytes"]) / 2 ** 20, samples=r)
    print(json.dumps({k: v for k, v in out.items() if k not in ("shared", "per_env")}))
    for plan in ("shared", "per_env"):
        print(plan, json.dumps({k: v for k, v in out[plan].items() if k != "samples"}))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
