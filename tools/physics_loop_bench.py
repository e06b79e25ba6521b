"""Device time per env-step of the loop a simulator runs, obs_t -> policy -> pre_physics_step(a_t) -> physics ->
post_physics_step() -> obs_{t+1}, with a stand-in for physics that only swaps the view's pose / joint tensors between the halves:
  (a) reference  pre_physics_step_device + post_physics_step   (the reference-shaped sequence of library calls)
  (b) fused      pre_physics_step_fused + post_physics_step_fused   (rvb_env_pre + rvb_env_post)
  (b16)          (b) with the packed fp16 observation (obs16_buf)
  (c) hot_step   hot_step(device_reset=True)   (rvb_env_pre + rvb_env_post with no physics between them, the reset half first;
                                                what bench.py times)
Benchmark world (200 m, K = 200, 2000 stones), curriculum level 2, device-side reset on, one task per size.  The arms alternate
round by round on the same task, so they see the same state distribution and the same clocks.  Every window is bracketed by CUDA
events on the task's stream after a synchronise, so host time that holds the stream back is part of what is measured.

  python tools/physics_loop_bench.py [--envs 4096,131072] [--steps 20] [--warmup 3] [--rounds 5] [--out FILE]
prints one JSON line (and writes it to FILE)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ARMS = ("reference", "fused", "fused_obs16", "hot_step")


def card():
    """Name, power limit and SM clocks of GPU 0, read now (nvidia-smi queries only)."""
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), [v.strip() for v in out.split(",")]))
    except (OSError, subprocess.SubprocessError) as e:
        return {"name": torch.cuda.get_device_name(0), "error": str(e)}


def run_size(R, w, N, args):
    dev = torch.device("cuda:0")
    n_sets = 3
    states = [{k: v.to(dev) for k, v in R.synth.make_env_state(w, N, seed=100 + s).items()} for s in range(n_sets)]
    task = R.synth.make_task(w, {k: v.cpu() for k, v in states[0].items()}, device="cuda:0", level=2, num_envs_total=N,
                             compact_terrain=True)
    view = task._rover
    obs16 = torch.zeros((N, task.num_observations - 4), dtype=torch.float16, device=dev)

    def physics(i):
        s = states[i % n_sets]
        view.pos, view.quat, view.joints = s["pos"], s["quat"], s["joints"]
        return s["actions"]

    def step(arm, i):
        act = physics(i)
        if arm == "hot_step":
            task.hot_step(act, device_reset=True)
            return
        if arm == "reference":
            task.pre_physics_step_device(act)
            physics(i + 1)
            task.post_physics_step()
        else:
            task.pre_physics_step_fused(act)
            physics(i + 1)
            task.post_physics_step_fused()

    ms = {a: [] for a in ARMS}
    launches = {}
    i = 0
    for r in range(args.rounds):
        for arm in ARMS:
            task.obs16_buf = obs16 if arm == "fused_obs16" else None
            for _ in range(args.warmup):
                step(arm, i)
                i += 1
            torch.cuda.synchronize()
            l0 = R._lib.launch_count
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.steps):
                step(arm, i)
                i += 1
            e1.record()
            torch.cuda.synchronize()
            ms[arm].append(e0.elapsed_time(e1) / args.steps)
            launches[arm] = (R._lib.launch_count - l0) / args.steps
    task.obs16_buf = None
    res = {}
    for arm in ARMS:
        med = statistics.median(ms[arm])
        res[arm] = {"ms_per_step_median": round(med, 4), "ms_per_step_min": round(min(ms[arm]), 4),
                    "ms_per_step_max": round(max(ms[arm]), 4), "env_steps_per_s": round(N / (med * 1e-3)),
                    "library_kernel_launches_per_step": launches[arm], "rounds_ms": [round(v, 4) for v in ms[arm]]}
    del task
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", default="4096,131072")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("physics_loop_bench.py: no CUDA device -- there is no CPU path")
    import isaac_rover_b200 as R
    before = card()
    w = R.synth.make_world(length=200.0, nv=708, K=200, n_stones=2000, seed=42, build_index=None)
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device="cuda:0")
    w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, w.K, device="cuda:0")
    t0 = time.time()
    sizes = {}
    for n in (int(v) for v in args.envs.split(",")):
        sizes[str(n)] = run_size(R, w, n, args)
    out = {"tool": "tools/physics_loop_bench.py", "card_before": before, "card_after": card(),
           "torch": torch.__version__, "cuda": torch.version.cuda, "curriculum_level": 2, "device_reset": True,
           "world": {"length_m": 200.0, "K": 200, "stones": 2000}, "steps": args.steps, "warmup": args.warmup,
           "rounds": args.rounds, "seconds": round(time.time() - t0, 1), "sizes": sizes}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
