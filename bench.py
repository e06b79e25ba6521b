#!/usr/bin/env python
"""Benchmark of the rover hot path (BASELINE.json metric: env-steps/s and heightmap rays/s).

  python bench.py --gpus N --steps K --warmup W            # this repo (hand-written sm_100a kernels)
  python bench.py --impl reference --gpus N --steps K ...  # the UNMODIFIED reference's torch code on the host cores
  python bench.py ... --dump-outputs DIR                   # also write the last timed step's outputs as DIR/<name>.npy, so
                                                           # that two builds can be compared on identical seeded inputs

Workload (BASELINE.json configs[3], one rank's share = configs[2] plus the device-side reset path): 131,072 envs per GPU
(`--envs`; 65,536 when the GPU has less than 60 GB free; `--envs 4096` = configs[1]), full dense+sparse heightmap (1634
rays/env, K=200 candidates/ray) on a synthetic 200 x 200 m, ~1M-triangle terrain (708^2 heightfield), big_rock_layer
collision, stone_info goal validation for the envs that reset, Ackermann kinematics, reward/reset terms.  One "step" = one
pass of the hot path over all envs: the reset half of pre_physics_step on the device (rover.py:356-361) + its action half +
post_physics_step (RoverTask.hot_step(device_reset=True)), PhysX excluded.  Multi-GPU: envs sharded by index (weak scaling),
terrain replicated, one NCCL all-reduce of the 16-entry statistics vector per step.
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

P_RAYS = 1634
ALGO_BYTES_PER_ENV_STEP = 665196          # SURVEY.md 8(d): index rows 785*K*4 + unique triangles + inputs + outputs
PEAKS_FILE = os.path.join(ROOT, "MEASURED_PEAKS.json")
FALLBACK_HBM_GBS = 6650.0                 # /opt/skills/guides/B200_PROFILING.md fallback
METRIC = "env-steps/sec (obs+kinematics+reward)"
C4_ENVS_PER_GPU = 131072                  # BASELINE.json configs[3]: 1,048,576 envs over 8 GPUs
DUMP_ENVS = 8192                          # --dump-outputs: envs sampled; their obs rows alone are 8192 x 1750 f32 = 57 MB
DUMP_MAX_BYTES = 64 * 10 ** 6


_JSON_FD = None


def claim_stdout():
    """Everything that libraries print to stdout while the benchmark runs (NCCL's "NCCL version ..." banner, for one) goes to
    stderr; the ONE JSON line is written to the real stdout by emit()."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def hbm_peak():
    try:
        return float(json.load(open(PEAKS_FILE))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def workload_config(envs_per_gpu, world_size, K=200, length=200.0, nv=708):
    """The `config` object of BOTH arms (this repo's and `--impl reference`): the workload, nothing measured."""
    ntri = 2 * (nv - 1) * (nv - 1)
    cfg_name = {4096: "configs[1]", 65536: "configs[2]", C4_ENVS_PER_GPU: "configs[3] (1,048,576 envs / 8 GPUs), one rank's share = configs[2] at twice the envs"}
    return {"workload": "%d envs/GPU, 1634 rays/env, K=%d, %gx%g m %d-triangle synthetic terrain + big_rock_layer collision + "
                        "stone_info goal validation of resetting envs + Ackermann + reward/reset; BASELINE.json %s"
                        % (envs_per_gpu, K, length, length, ntri, cfg_name.get(envs_per_gpu, "(custom size)")),
            "envs_per_gpu": envs_per_gpu, "total_envs": envs_per_gpu * world_size, "rays_per_env": P_RAYS, "K": K,
            "index_cells": int(round(length / 0.1)) ** 2,
            "l2": "inputs larger than L2: 3 pose sets cycled, %.1f GB of index rows touched per step, index %.1f GB"
                  % (envs_per_gpu * 785 * K * 4 / 1e9, int(round(length / 0.1)) ** 2 * K * 4 / 1e9),
            "parallelism": "env shards x%d, terrain replicated, 1 all-reduce of 16 f64 per step" % world_size}


class ClockSampler:
    """SM clock + throttle reasons sampled every 10 ms during the timed regions: NVML in a background thread of this
    process (what `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` reads, without spawning a poller process
    that contends with the benchmark for the driver); falls back to an `nvidia-smi -lms 50` child if NVML is missing.
    Constructed on EVERY rank, before the barrier that precedes the timed region (NVML initialisation takes milliseconds)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc, self.thread, self.sm, self.reasons, self.mx = None, None, [], set(), None
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            uuid = None
            try:
                uuid = torch.cuda.get_device_properties(index).uuid          # CUDA_VISIBLE_DEVICES-proof
                h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + str(uuid)).encode())
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(index)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
            self.stop_flag = threading.Event()
            self.active = threading.Event()

            def poll():
                while not self.stop_flag.is_set():
                    if self.active.is_set():
                        try:
                            self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                            for name, b in bits.items():
                                if r & b:
                                    self.reasons.add(name)
                        except Exception:
                            pass
                    self.stop_flag.wait(0.01)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                                          "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def start(self):
        if self.thread is not None:
            self.active.set()

    def stop(self):
        if self.thread is not None:
            self.stop_flag.set()
            self.thread.join(timeout=2)
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx, "samples": len(self.sm),
                    "reasons": sorted(self.reasons), "source": "NVML, 10 ms period, in-process thread"}
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi -lms 50"}


# ------------------------------------------------------------------------------------------------ reference arm
def reference_world(args):
    """The benchmark's world with the index tensors in the reference's asset format ([K,G,G] int32 on the host).  The index of
    the 200 m world (4 M cells x 1 M triangles) cannot be built by CPU brute force in any reasonable time, so the synthetic asset
    is produced with the GPU index builder when a GPU is present (input synthesis, like the terrain itself -- nothing of the
    timed path); without a GPU the world is a 24 m crop of the same mesh density (the reference's per-env cost does not depend
    on the map extent)."""
    import isaac_rover_b200 as R
    from isaac_rover_b200 import synth
    if torch.cuda.is_available():
        w = synth.make_world(length=args.length, nv=args.nv, K=args.K, n_stones=args.stones, seed=42, build_index=None)
        w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device="cuda:0").cpu()
        w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, w.K, device="cuda:0").cpu()
        torch.cuda.empty_cache()
        return w, "%gx%g m world, %d triangles (the benchmark's)" % (args.length, args.length, w.triangles.shape[0])
    w = synth.make_world(length=24.0, nv=86, K=args.K, n_stones=30, seed=42, build_index="cpu")
    return w, "24 m crop of the benchmark's mesh density (no GPU here to synthesise the 200 m index)"


def time_reference(args, device, n_envs, steps, warmup):
    """-> (seconds per step, kind, description).  kind = "reference": the unmodified reference's classes (oracle/ref_harness.py,
    from baseline/_ref or /root/reference); "port": the oracle restatement, only if no reference tree is present."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from isaac_rover_b200 import synth
    w, wdesc = reference_world(args)
    st = synth.make_env_state(w, n_envs, seed=100, margin=6.0)
    st = {k: v.to(device) for k, v in st.items()}
    import ref_harness
    root = ref_harness.reference_root()
    cuda = device != "cpu"

    def sync():
        if cuda:
            torch.cuda.synchronize()
    if root is not None:
        ns = ref_harness.load("cpu" if not cuda else "cuda")
        fake = ref_harness.make_fake_task(ns, w, st, level=2, device=device)
        w.map_indices = w.rock_indices = None

        def step():
            ref_harness.reference_step(ns, fake, st)
        kind, what = "reference", "unmodified reference classes from %s" % os.path.relpath(root, ROOT)
    else:
        import rover_oracle as O
        pat, ci, fi = O.heightmap_pattern()
        assets = dict(pattern=pat, coarse_idx=ci, fi=fi, fine_idx=fi, map_indices=w.map_indices, triangles=w.triangles,
                      vertices=w.vertices, rock_indices=w.rock_indices, rock_triangles=w.rock_triangles,
                      rock_vertices=w.rock_vertices, shift=torch.tensor([0, 0, 0.0]))
        assets = {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in assets.items()}

        def step():
            O.full_step(assets, st, env_chunk=min(n_envs, 128))
        kind, what = "port", "oracle restatement (no reference tree on this box)"
    for _ in range(warmup):
        step()
    sync()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        step()
        sync()
        ts.append(time.perf_counter() - t0)
    return statistics.median(ts), kind, "%s; %s; %d envs x %d rays x K=%d per step, %d warm-up + %d timed steps (median)" % (
        what, wdesc, n_envs, P_RAYS, args.K, warmup, steps)


def run_reference(args, rank, world):
    """`--impl reference`: BASELINE.json configs[0] -- the reference's torch path on the host cores (all of them), 64 envs per
    step on the benchmark's world.  Rank 0 only."""
    if rank != 0:
        return
    device = args.ref_device
    n = args.ref_envs
    if device == "cpu":
        torch.set_num_threads(os.cpu_count())
        budget = 30                                    # keep the whole run within a few minutes (~5 s per 64-env step)
        if args.steps + args.warmup > budget:
            n = max(8, n * budget // (args.steps + args.warmup))
    t, kind, sample = time_reference(args, device, n, args.steps, args.warmup)
    v = n / t
    cores = torch.get_num_threads() if device == "cpu" else 0
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "env-steps/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": workload_config(args.envs or C4_ENVS_PER_GPU, world, args.K, args.length, args.nv),
            "rays_per_s": v * P_RAYS, "device": device, "sample_envs": n,
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)


def reference_subprocess(device, envs, steps, warmup, timeout=420):
    """The reference arm in a child process (its CPU recipe re-points torch defaults that this process must not see)."""
    cmd = [sys.executable, os.path.abspath(__file__), "--impl", "reference", "--ref-device", device, "--ref-envs", str(envs),
           "--steps", str(steps), "--warmup", str(warmup)]
    env = dict(os.environ)
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT"):
        env.pop(k, None)
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=timeout, env=env)
    for ln in reversed(r.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)
    raise RuntimeError("reference arm failed: " + (r.stderr or r.stdout)[-300:])


def time_policy_epilogue(R, obs, steps=20, warmup=3):
    """SURVEY.md 8f-3, reported beside the step (not part of `value`): actor + critic inference on the step's obs_buf through
    rvb_policy_forward, and the same two networks as eager torch fp32 (cuBLAS) on this GPU for comparison."""
    import torch.nn.functional as F
    N = obs.shape[0]
    net = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], "leakyrelu")
    info = R.model.ObserverationInfo(4, 634, 1112, 0)
    actor = R.model.StochasticActorHeightmap(1750, 2, net, info, device=obs.device)
    critic = R.model.DeterministicHeightmap(1750, 2, net, info, device=obs.device)
    out_a = torch.empty((N, 2), dtype=torch.float32, device=obs.device)
    out_c = torch.empty((N, 1), dtype=torch.float32, device=obs.device)

    def ours():
        R.model.compute_pair(actor, critic, obs, out_a, out_c)

    def ours_single():
        actor._forward(obs, out_a)

    def eager_net(sd, tanh):
        sd = {k: v.to(obs.device) for k, v in sd.items()}

        def chain(x, prefix, n):
            for i in range(n):
                x = F.leaky_relu(F.linear(x, sd["%s.%d.layer.0.weight" % (prefix, i)], sd["%s.%d.layer.0.bias" % (prefix, i)]))
            return x

        def fwd():
            x = torch.cat((obs[:, 0:4], chain(obs[:, 4:638], "encoder0.encoder", 2), chain(obs[:, 638:1750], "encoder1.encoder", 2)), dim=1)
            x = F.linear(chain(x, "network", 3), sd["network.3.weight"], sd["network.3.bias"])
            return torch.tanh(x) if tanh else x
        return fwd
    ea, ec = eager_net(actor.state_dict(), True), eager_net(critic.state_dict(), False)

    def timed(fn):
        for _ in range(warmup):
            fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / steps
    ms = timed(ours)
    ms_single = timed(ours_single)
    ms_eager = timed(lambda: (ea(), ec()))
    err = max((out_a - ea()).abs().max().item(), (out_c - ec()).abs().max().item())
    flops = 2 * 2 * N * (634 * 80 + 1112 * 80 + 2 * 80 * 60 + 124 * 256 + 256 * 160 + 160 * 128 + 128 * 2)
    lib = R._lib.load()
    prev = lib.rvb_policy_variant(1)                 # the round-1 fp32 FFMA2 kernel, for comparison
    try:
        ms_ffma = timed(ours)
    finally:
        lib.rvb_policy_variant(prev)
    return {"ms": ms, "envs_per_s": N / ms * 1e3, "fp32_equivalent_tflops": flops / ms / 1e9, "torch_eager_fp32_ms": ms_eager,
            "ffma2_kernel_ms": ms_ffma, "max_abs_diff_vs_torch": err, "launches": 2, "actor_alone_ms": ms_single,
            "what": "actor + critic (encoders [80,60] x2, mlp [256,160,128], model.py:152-241) on the step's obs_buf f32 [%d,1750] through "
                    "rvb_policy_forward_pair: two launches, tcgen05 kind::tf32 MMAs with hi + lo split operands (fp32-grade), accumulators "
                    "in TMEM (policy_l1_tc_kernel + policy_tail_tc_kernel); not included in `value`" % N}


# ------------------------------------------------------------------------------------------------ B200 arm
def last_step_outputs(task, stats):
    """What the last timed step returned to its caller (hot_step: obs, rew, reset, extras), the joint targets it computed for
    the simulator and the step's reduced statistics, as host arrays (float32; float64 for the statistics and for integers).
    The per-env arrays keep a fixed, seeded sample of DUMP_ENVS envs, sorted; `env_ids` holds their indices."""
    N = task.num_envs
    ids = torch.randperm(N, generator=torch.Generator().manual_seed(0))[:DUMP_ENVS].sort().values
    ids_d = ids.to(task.obs_buf.device)
    per_env = {"obs": task.obs_buf, "rew": task.rew_buf, "reset": task.reset_buf,
               "joint_position_targets": task.joint_position_targets, "joint_velocity_targets": task.joint_velocity_targets}
    per_env.update({"extras_" + k: v for k, v in task.extras.items()})
    out = {"env_ids": ids.double().numpy(), "stats": stats.double().cpu().numpy()}
    for name, t in per_env.items():
        t = t[ids_d].cpu()
        out[name] = (t.float() if t.is_floating_point() and t.dtype != torch.float64 else t.double()).numpy()
    nbytes = sum(a.nbytes for a in out.values())
    if nbytes > DUMP_MAX_BYTES:
        raise RuntimeError("--dump-outputs: %d bytes exceed the %d-byte limit" % (nbytes, DUMP_MAX_BYTES))
    return out


def run_b200(args, rank, world, local):
    import isaac_rover_b200 as R
    from isaac_rover_b200 import synth
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py: no CUDA device -- this arm has no CPU path")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    numa_cpus = None if args.no_numa else R.dist.bind_to_gpu_numa(local)      # before any pinned buffer exists
    N = args.envs
    if not N:
        free_b, _ = torch.cuda.mem_get_info(dev)
        N = C4_ENVS_PER_GPU if free_b > 60e9 else 65536
    w = synth.make_world(length=args.length, nv=args.nv, K=args.K, n_stones=args.stones, seed=42, build_index=None)
    t0 = time.perf_counter()
    w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device=dev)
    w.rock_indices = R.build_knn_index(w.rock_triangles, w.rock_vertices, w.G, w.res, w.K, device=dev)
    torch.cuda.synchronize()
    t_index = time.perf_counter() - t0
    n_sets = 3
    states = [synth.make_env_state(w, N, seed=100 + s, env_offset=rank * N) for s in range(n_sets)]
    # compact_terrain: the heightmap layer keeps no K-contiguous copy of the index (rvb_terrain_release_index) -- the production
    # kernels never read it; `setup.heightmap_layer_gb` is what the layer then holds, `index_gb` the reference's own tensor
    task = synth.make_task(w, states[0], device=str(dev), level=2, num_envs_total=N * world, compact_terrain=not args.full_layer and args.variant in (0, 3))
    task.env_offset = rank * N
    w.map_indices = w.rock_indices = None          # the layers own K-contiguous copies
    torch.cuda.empty_cache()
    dstates = [{k: v.to(dev) for k, v in s.items()} for s in states]
    view = task._rover

    def set_state(i):
        s = dstates[i % n_sets]
        view.pos, view.quat, view.joints = s["pos"], s["quat"], s["joints"]
        return s["actions"]

    reducer = R.dist.StatsReducer(depth=4)
    device_reset = not args.no_reset

    def step(i):
        task.hot_step(set_state(i), fused=not args.unfused, device_reset=device_reset)
        if args.sync_reduce:
            R.dist.reduce_stats(task.stats)
        else:
            reducer.submit(task.stats)          # asynchronous all-reduce of the 16 sums (off the critical path)

    task.Camera.variant = args.variant
    clocks = ClockSampler(local)                # every rank, BEFORE the barrier (pynvml import + nvmlInit take milliseconds)
    lib = R._lib.load()
    for i in range(args.warmup):
        step(i)
    torch.cuda.synchronize()
    task.reset_counters.zero_()
    task.Camera.timing = []
    lib.rvb_timing_enable(1)
    launches0 = R._lib.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if rank == 0:
        clocks.start()
    R.dist.barrier()
    torch.cuda.synchronize()
    e0.record()
    for i in range(args.steps):
        step(args.warmup + i)
    if not args.sync_reduce:
        reducer.result((reducer.i - 1) % reducer.depth)       # the timed region ends when the last reduction has landed
    e1.record()
    torch.cuda.synchronize()
    R.dist.barrier()
    launches = R._lib.launch_count - launches0
    # taken before the passes below reuse the task's buffers
    dumped = None
    if args.dump_outputs and rank == 0:
        dumped = last_step_outputs(task, task.stats if args.sync_reduce else reducer.result((reducer.i - 1) % reducer.depth))
    dt = R.dist.max_over_ranks(e0.elapsed_time(e1) * 1e-3, dev)
    reset_counts = task.reset_counters.cpu().tolist()
    ray_ms = [a.elapsed_time(b) for a, b in task.Camera.timing]
    task.Camera.timing = None
    if not ray_ms:          # fused step: the library timed the ray-cast itself (CUDA events on the launching stream)
        import ctypes
        buf = (ctypes.c_float * (args.steps + 8))()
        n_t = lib.rvb_timing_read(buf, args.steps + 8)
        ray_ms = [buf[i] for i in range(max(n_t, 0))]
    lib.rvb_timing_enable(0)
    ray_s = R.dist.max_over_ranks(sum(ray_ms) / len(ray_ms) * 1e-3, dev)
    # ---- end to end through the host-buffer API (H2D + hot path + D2H every step)
    hstates = [{k: v.pin_memory() for k, v in s.items() if k in ("pos", "quat", "joints", "actions")} for s in states]

    def run_e2e(packed):
        """every step: inputs copied from pinned host memory, results (obs, rew, reset) read back and touched on the host;
        two slots, so the read-back of step i overlaps the kernels of step i+1"""
        pipe = R.HostPipeline(task, packed_obs=packed, device_reset=device_reset)
        for i in range(max(args.warmup, 3)):
            h = hstates[i % n_sets]
            pipe.step(h["pos"], h["quat"], h["joints"], h["actions"])
        torch.cuda.synchronize()
        R.dist.barrier()
        t0 = time.perf_counter()
        prev, checksum = None, 0.0

        def touch(res):
            rew_h, reset_h = res[-2], res[-1]
            return float(rew_h[0]) + float(res[-3][-1, -1]) + int(reset_h[0])
        for i in range(args.steps):
            h = hstates[i % n_sets]
            k = pipe.submit(h["pos"], h["quat"], h["joints"], h["actions"])
            if args.sync_reduce:
                R.dist.reduce_stats(task.stats)
            else:
                reducer.submit(task.stats)
            if prev is not None:
                checksum += touch(pipe.result(prev))
            prev = k
        checksum += touch(pipe.result(prev))
        if not args.sync_reduce:
            reducer.result((reducer.i - 1) % reducer.depth)
        torch.cuda.synchronize()
        dt_ = R.dist.max_over_ranks(time.perf_counter() - t0, dev)
        task.obs16_buf = None
        h2d, d2h = pipe.h2d_bytes, pipe.d2h_bytes
        pipe.close()
        return dt_, h2d, d2h, checksum
    # the dominant kernel by itself (no rock kernel sharing the SMs): the same launches as in the step, timed with CUDA events
    def time_raycast_alone():
        reps = max(3, min(args.steps, 10))
        pos, quat = view.get_world_poses()
        eul = R.tensor_quat_to_eul(quat)
        for _ in range(2):
            task.Camera.get_depths(pos, eul, obs=task.obs_buf, want_pt=False)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record()
        for i in range(reps):
            s_ = dstates[i % n_sets]
            task.Camera.get_depths(s_["pos"], eul, obs=task.obs_buf, want_pt=False)
        b.record()
        torch.cuda.synchronize()
        return R.dist.max_over_ranks(a.elapsed_time(b) / reps * 1e-3, dev)
    ray_alone_s = time_raycast_alone()
    dt_e2e, h2d_b, d2h_b, checksum = run_e2e(False)
    dt_e2e_p, h2d_bp, d2h_bp, checksum_p = run_e2e(True)
    clk = clocks.stop()
    if rank != 0:
        return
    total_envs = N * world
    value = total_envs * args.steps / dt
    peak, peak_src = hbm_peak()
    achieved = ALGO_BYTES_PER_ENV_STEP * N / ray_s / 1e9
    traffic, issue = None, None
    tf = os.path.join(ROOT, "profiles", "raycast_traffic.json")
    if os.path.exists(tf):
        try:
            prof = json.load(open(tf))
            # the capture is only quoted for the build it was taken from: raycast_traffic.json carries the source hash
            same_build = prof.get("source_hash") == R._build.raycast_hash()
            traffic = prof.get("dram_bytes_per_launch") if same_build else None
            if traffic is not None:
                traffic = traffic / prof["envs_per_launch"] * N          # per launch of THIS run (traffic scales with the envs)
            # the resource that actually binds the kernel (DESIGN.md 4.1): warp-instruction issue slots.  Instruction count per
            # env from the ncu capture (smsp__inst_executed.sum), time measured live, clock sampled live
            if same_build:
                wi = prof["warp_instructions_per_launch"] / prof["envs_per_launch"] * N
                clk_hz = float(clk["sm_mhz"]) * 1e6 if (clk and clk.get("sm_mhz")) else 1.965e9      # median SM clock under load
                issue = {"warp_inst_per_launch": wi, "source": prof.get("source"), "sm_clock_hz": clk_hz,
                         "peak_warp_inst_per_s": 148 * 4 * clk_hz, "achieved_warp_inst_per_s": wi / ray_s,
                         "frac": wi / ray_s / (148 * 4 * clk_hz)}
            else:
                issue = {"unavailable": "profiles/raycast_traffic.json was captured from another build of the kernels"}
        except Exception:
            traffic, issue = None, None
    cfg = workload_config(N, world, w.K, w.length, args.nv)
    line = {"metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16", "data": "synthetic",
            "config": cfg,
            "setup": {"raycast_variant": args.variant, "fused_step": not args.unfused, "index_build_s": round(t_index, 3),
                      "rock_triangles": int(w.rock_triangles.shape[0]), "stones": int(w.stone_info.shape[0]),
                      "stats_reduction": "compute stream" if args.sync_reduce else "asynchronous, NCCL stream",
                      "device_reset_in_step": device_reset, "cpus_after_numa_binding": numa_cpus,
                      "heightmap_layer_gb": round(task.Camera.layer.bytes() / 1e9, 3), "heightmap_layer_keeps_index_copy": task.Camera.layer.has_index,
                      "index_gb": round(w.K * w.G * w.G * 4 / 1e9, 3), "rock_layer_gb": round(task.Rock_detector.layer.bytes() / 1e9, 3),
                      "resets_per_step": reset_counts[0] / max(args.steps, 1), "goals_drawn_per_step": reset_counts[1] / max(args.steps, 1),
                      "reset_rate": reset_counts[0] / max(args.steps, 1) / N},
            "rays_per_s": value * P_RAYS,
            # (ray, candidate) tests the reference evaluates for the same output: (1634 heightmap + 26 rock rays) x K per env-step
            "reference_equivalent_pair_tests_per_s": value * (P_RAYS + 26) * w.K,
            "raycast_ms": ray_s * 1e3,
            "raycast_share_of_step": ray_s / (dt / args.steps),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": ALGO_BYTES_PER_ENV_STEP * N,
                         "kernel_alone": {"ms": ray_alone_s * 1e3, "achieved": ALGO_BYTES_PER_ENV_STEP * N / ray_alone_s / 1e9,
                                          "frac": ALGO_BYTES_PER_ENV_STEP * N / ray_alone_s / 1e9 / peak,
                                          "note": "the same launch without the rock-collision kernel running beside it (in the step the "
                                                  "two share the SMs and `achieved` is measured around the ray-cast's launches)"},
                         "kernel": "heightmap ray-cast (Camera.get_depths)",
                         "note": "contractual HBM figure on the reference-format algorithmic bytes; the kernel is bound by "
                                 "instruction issue, see issue_slots", "issue_slots": issue},
            # headline end-to-end number: the host pipeline returning the reference's output type, obs_buf f32 [N,1750]
            # (rover.py:320-325); e2e_packed_obs is the same loop with the heightmap columns read back as the fp16 values they
            # are (half the bytes; HostPipeline.obs_f32() widens them on the host)
            "e2e": {"value": total_envs * args.steps / dt_e2e, "unit": "env-steps/s", "h2d_bytes_per_step": h2d_b * world,
                    "d2h_bytes_per_step": d2h_b * world, "ms_per_step": dt_e2e / args.steps * 1e3,
                    "api": "HostPipeline.submit/result (2 slots: read-back of step i overlaps step i+1; inputs uploaded from "
                           "pinned host memory every step; obs f32 [N,1750], rew f32 [N], reset i64 [N] read back)",
                    "checksum": checksum},
            "e2e_packed_obs": {"value": total_envs * args.steps / dt_e2e_p, "unit": "env-steps/s", "h2d_bytes_per_step": h2d_bp * world,
                               "d2h_bytes_per_step": d2h_bp * world, "ms_per_step": dt_e2e_p / args.steps * 1e3,
                               "api": "HostPipeline(packed_obs=True): obs = f32 [N,4] proprioceptive + f16 [N,1746] heightmap "
                                      "columns, lossless", "checksum": checksum_p},
            "gpu_launches": launches,
            "clocks": clk}
    act0 = dstates[0]["actions"]
    if world == 1 and not args.no_cpu:
        del dstates, hstates
        torch.cuda.empty_cache()
        try:
            ref = reference_subprocess("cpu", args.ref_envs, 2, 1)
            line["cpu_baseline"] = ref["cpu_baseline"]
        except Exception as e:          # a baseline, never a reason to lose the bench line
            line["cpu_baseline"] = {"unavailable": str(e)[:300]}
        try:
            ref = reference_subprocess("cuda:0", 512, 3, 1)
            line["torch_eager_gpu_baseline"] = {"value": ref["value"], "unit": "env-steps/s", "kind": ref["cpu_baseline"]["kind"],
                                                "sample": ref["cpu_baseline"]["sample"] + " -- the reference's own deployment: "
                                                "eager torch on cuda:0 (rover.py:90), N = 512 (its default)"}
        except Exception as e:
            line["torch_eager_gpu_baseline"] = {"unavailable": str(e)[:300]}
    if world == 1:
        try:
            # a real observation for the consumer: the host pipelines left task.obs_buf pointing at their own (packed: empty) slots
            task.obs16_buf = None
            task.obs_buf = torch.zeros((N, task.num_observations), device=dev)
            task.hot_step(act0)
            torch.cuda.synchronize()
            line["policy_epilogue"] = time_policy_epilogue(R, task.obs_buf)
        except Exception as e:          # reported beside the step, never a reason to lose the bench line
            line["policy_epilogue"] = {"unavailable": str(e)[:200]}
    if dumped is not None:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in dumped.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=0, help="envs per GPU (default 131072 = BASELINE.json configs[3]'s share; 4096 = configs[1])")
    ap.add_argument("--length", type=float, default=200.0)
    ap.add_argument("--nv", type=int, default=708)
    ap.add_argument("--K", type=int, default=200)
    ap.add_argument("--stones", type=int, default=2000)
    ap.add_argument("--variant", type=int, default=0)
    ap.add_argument("--ref-envs", type=int, default=64, help="envs per step of the reference arm (BASELINE.json configs[0]: 64)")
    ap.add_argument("--ref-device", default="cpu", help="reference arm: cpu (the baseline) or cuda:0 (its own eager deployment)")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-reset", action="store_true", help="leave the device-side reset path out of the step")
    ap.add_argument("--full-layer", action="store_true", help="the heightmap layer keeps its K-contiguous index copy (+3.2 GB; what the cross-check variants 1 / 2 read)")
    ap.add_argument("--no-numa", action="store_true", help="do not bind the process to the CPUs local to its GPU")
    ap.add_argument("--unfused", action="store_true", help="one library call per reference call instead of rvb_env_step")
    ap.add_argument("--sync-reduce", action="store_true", help="all-reduce the statistics on the compute stream every step")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (rank 0's "
                    "envs; obs, rew, reset, extras and joint targets of %d seeded sample envs, the reduced statistics)" % DUMP_ENVS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    args.warmup = max(args.warmup, 1 if args.impl == "reference" else 3)
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    claim_stdout()
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import isaac_rover_b200 as R
    rank, world, local = R.dist.init_from_env()
    try:
        run_b200(args, rank, world, local)
    finally:
        if world > 1 and torch.distributed.is_initialized():
            torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
