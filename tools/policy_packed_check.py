"""GPU timing of the policy + value pair on the step's packed observation (rvb_policy_forward_packed) against the f32 rows.

At N = 4096 and 131,072 envs with the shipped widths (S = 634, D = 1112, actor head 2 + tanh, critic head 1), in one process,
alternating the three and after a warm-up, CUDA events around `ITERS` back-to-back calls of
  (a) compute_pair on the f32 rows [N, 1750],
  (b) compute_pair on the packed pair (proprio f32 [N, 4] as the strided view obs[:, :4], heightmap f16 [N, 1746]),
  (c) what a caller of (a) has to do with a packed step today: torch.cat((proprio, heightmap.float()), 1), then (a).
(b) must return the bits of (a) on the widened rows.  The f32 rows are 28.7 MB at 4096 envs (L2-resident after the first call)
and 917 MB at 131,072 (read from HBM).  Prints the card's name and power limit with the numbers.
"""
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import isaac_rover_b200 as R  # noqa: E402

ITERS, ROUNDS, WARMUP = 20, 7, 5


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.TimeoutExpired):
        q = "nvidia-smi unavailable"
    return "%s | nvidia-smi: %s" % (torch.cuda.get_device_name(0), q)


def main():
    if not torch.cuda.is_available():
        raise SystemExit("policy_packed_check: needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(1)
    net = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], "leakyrelu")
    info = R.model.ObserverationInfo(4, 634, 1112, 0)
    actor = R.model.StochasticActorHeightmap(1750, 2, net, info, device="cuda:0")
    critic = R.model.DeterministicHeightmap(1750, 1, net, info, device="cuda:0")
    print("card:", card())
    print("policy variant %d (2 = tensor-core path), %d rounds x %d calls per mode, median of the rounds" % (
        R._lib.load().rvb_policy_variant(-1), ROUNDS, ITERS))
    for N in (4096, 131072):
        obs = torch.rand(N, 1750, device="cuda") * 2 - 1
        h16 = (torch.rand(N, 1746, device="cuda") * 8).half()
        obs[:, 4:] = h16.float()
        proprio = obs[:, :4]
        out = (torch.empty(N, 2, device="cuda"), torch.empty(N, 1, device="cuda"))
        modes = {
            "a_f32_rows": lambda: R.model.compute_pair(actor, critic, obs, *out),
            "b_packed": lambda: R.model.compute_pair(actor, critic, (proprio, h16), *out),
            "c_widen_then_f32": lambda: R.model.compute_pair(actor, critic, torch.cat((proprio, h16.float()), 1), *out),
        }
        ref = [t.clone() for t in R.model.compute_pair(actor, critic, obs)]
        got = R.model.compute_pair(actor, critic, (proprio, h16))
        same = torch.equal(got[0], ref[0]) and torch.equal(got[1], ref[1])
        for fn in modes.values():
            for _ in range(WARMUP):
                fn()
        torch.cuda.synchronize()
        times = {k: [] for k in modes}
        for r in range(ROUNDS):
            order = list(modes)[r % 3:] + list(modes)[:r % 3]
            for k in order:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(ITERS):
                    modes[k]()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / ITERS)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        hm_f32, hm_f16 = N * 1746 * 4 / 1e9, N * 1746 * 2 / 1e9
        print("N %6d: (a) f32 rows %.4f ms | (b) packed %.4f ms | (c) widen + f32 %.4f ms | (b)/(a) %.3f (b)/(c) %.3f | "
              "(b) bit-identical to (a): %s | heightmap bytes per pair f32 %.3f GB, f16 %.3f GB" % (
                  N, med["a_f32_rows"], med["b_packed"], med["c_widen_then_f32"], med["b_packed"] / med["a_f32_rows"],
                  med["b_packed"] / med["c_widen_then_f32"], same, hm_f32, hm_f16))
        print("         spread (min..max over rounds): " + ", ".join("%s %.4f..%.4f" % (k, min(v), max(v)) for k, v in times.items()),
              flush=True)
        if not same:
            raise SystemExit("policy_packed_check: the packed call differs from the f32 rows")


if __name__ == "__main__":
    main()
