"""GPU timing of one teacher-data recorder call (rvb_teacher_record / rvb_teacher_record_packed) at the shipped row shape.

At N = 4096 and 131,072 envs (p = 4, 1746 heightmap columns), in one process, alternating the three arms after a warm-up, CUDA events
around `ITERS` back-to-back calls of
  (a) f32 rows:         rvb_teacher_record on obs_buf f32 [N, 1750] into an f32 block [T, N, 1753];
  (b) packed -> f32:    rvb_teacher_record_packed on (obs_buf[:, :4], obs16_buf f16 [N, 1746]) into the same f32 block;
  (c) packed -> packed: rvb_teacher_record_packed into a packed block, f32 [T, N, 7] + f16 [T, N, 1746].
Each call writes the next of T = 8 timesteps of its block, as the recorder does step after step; the observation is the same
buffer every call, as the step's output is (at 4096 envs it is L2-resident, as it is after a real step; at 131,072 it is not).
Bytes per call are computed from the shapes; their rate is given as a fraction of the B200's 7.7 TB/s HBM3e data-sheet bandwidth.
A torch.profiler pass after the timed rounds gives each arm's kernel time.  (b) and (c) must give the bits of (a).  Prints the
card's name and power limit with the numbers and writes them as JSON to --out.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import isaac_rover_b200 as R  # noqa: E402

T, ROUNDS, WARMUP = 8, 7, 10
ITERS = {4096: 200, 131072: 20}
HBM_BYTES_PER_S = 7.7e12
P, E = 4, 1746


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except (OSError, IndexError, subprocess.TimeoutExpired):
        q = "nvidia-smi unavailable"
    return "%s | nvidia-smi: %s" % (torch.cuda.get_device_name(0), q)


def bytes_per_call(N):
    lead_in = 4 + 8 + 4 * P                          # reset_info, actions, proprio
    return {"a_f32_rows": N * ((lead_in + 4 * E) + 4 * (3 + P + E)),
            "b_packed_to_f32": N * ((lead_in + 2 * E) + 4 * (3 + P + E)),
            "c_packed_to_packed": N * ((lead_in + 2 * E) + 4 * (3 + P) + 2 * E)}


def arms(lib, N):
    g = torch.Generator(device="cuda").manual_seed(N)
    obs16 = (torch.rand((N, E), device="cuda", generator=g) * 8).half()
    obs = torch.empty((N, P + E), device="cuda")
    obs[:, :P] = torch.rand((N, P), device="cuda", generator=g)
    obs[:, P:] = obs16.float()
    proprio = obs[:, :P]
    reset = (torch.rand(N, device="cuda", generator=g) < 0.5).float()
    actions = torch.rand((N, 2), device="cuda", generator=g) * 2 - 1
    block_a = torch.empty((T, N, 3 + P + E), device="cuda")
    block_b = torch.empty_like(block_a)
    head = torch.empty((T, N, 3 + P), device="cuda")
    hm = torch.empty((T, N, E), device="cuda", dtype=torch.float16)
    st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    ptr = lambda t: C.c_void_p(t.data_ptr())
    a_args = [(ptr(reset), ptr(actions), 2, ptr(obs), P + E, N, P + E, ptr(block_a[t]), 3 + P + E, st) for t in range(T)]
    b_args = [(ptr(reset), ptr(actions), 2, ptr(proprio), P + E, P, ptr(obs16), E, E, N, ptr(block_b[t]), 3 + P + E, None, 0, st)
              for t in range(T)]
    c_args = [(ptr(reset), ptr(actions), 2, ptr(proprio), P + E, P, ptr(obs16), E, E, N, ptr(head[t]), 3 + P, ptr(hm[t]), E, st)
              for t in range(T)]
    fa, fp = lib.rvb_teacher_record, lib.rvb_teacher_record_packed
    state = {"t": 0}

    def runner(fn, args):
        def run():
            t = state["t"] = (state["t"] + 1) % T
            if fn(*args[t]) != 0:
                raise RuntimeError(lib.rvb_last_error().decode())
        return run
    modes = {"a_f32_rows": runner(fa, a_args), "b_packed_to_f32": runner(fp, b_args), "c_packed_to_packed": runner(fp, c_args)}
    # bits: every timestep of all three blocks written from the same observation
    for t in range(T):
        for fn, args in ((fa, a_args), (fp, b_args), (fp, c_args)):
            assert fn(*args[t]) == 0, lib.rvb_last_error()
    torch.cuda.synchronize()
    same = (torch.equal(block_a.view(torch.int32), block_b.view(torch.int32))
            and torch.equal(head, block_a[:, :, :3 + P]) and torch.equal(hm.float(), block_a[:, :, 3 + P:]))
    return modes, same, (obs, obs16, block_a, block_b, head, hm)


def kernel_times(modes, n_calls=20):
    """Mean device time per call of each arm's kernel from a torch.profiler pass (its own pass, after the timed rounds)."""
    from torch.profiler import ProfilerActivity, profile
    out = {}
    for k, fn in modes.items():
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(n_calls):
                fn()
            torch.cuda.synchronize()
        tot = 0.0
        for e in prof.key_averages():
            if "teacher_record" in e.key:
                tot += getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0.0)
        out[k] = tot / n_calls / 1e3                  # us -> ms
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None, help="JSON file for the results")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("teacher_record_bench: needs a CUDA device")
    lib = R._lib.load()
    result = {"card": card(), "rounds": ROUNDS, "timesteps_rotated": T, "hbm_bytes_per_s_datasheet": HBM_BYTES_PER_S, "sizes": {}}
    print("card:", result["card"])
    for N in (4096, 131072):
        modes, same, keep = arms(lib, N)
        iters = ITERS[N]
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
                for _ in range(iters):
                    modes[k]()
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / iters)
        med = {k: sorted(v)[len(v) // 2] for k, v in times.items()}
        try:
            kern = kernel_times(modes)
        except Exception as ex:                       # the event times stand without it
            kern = {k: None for k in modes}
            print("profiler pass failed: %r" % (ex,))
        nbytes = bytes_per_call(N)
        row = {}
        for k in modes:
            row[k] = dict(ms_per_call=med[k], ms_min=min(times[k]), ms_max=max(times[k]), kernel_ms=kern[k], bytes=nbytes[k],
                          hbm_fraction=nbytes[k] / (med[k] * 1e-3) / HBM_BYTES_PER_S)
            print("N %6d %-19s %.4f ms/call (spread %.4f..%.4f, kernel %s ms) | %7.1f MB | %.2f TB/s = %.2f of 7.7 TB/s" % (
                N, k, med[k], min(times[k]), max(times[k]), "n/a" if kern[k] is None else "%.4f" % kern[k], nbytes[k] / 1e6,
                nbytes[k] / (med[k] * 1e-3) / 1e12, row[k]["hbm_fraction"]), flush=True)
        row["packed_to_packed_over_f32_rows"] = med["c_packed_to_packed"] / med["a_f32_rows"]
        row["packed_to_f32_over_f32_rows"] = med["b_packed_to_f32"] / med["a_f32_rows"]
        row["bits_equal"] = same
        print("N %6d (c)/(a) %.3f, (b)/(a) %.3f, blocks bit-identical: %s" % (N, row["packed_to_packed_over_f32_rows"],
                                                                          row["packed_to_f32_over_f32_rows"], same), flush=True)
        result["sizes"][str(N)] = row
        del modes, keep
        torch.cuda.empty_cache()
        if not same:
            raise SystemExit("teacher_record_bench: the packed blocks differ from the f32 rows")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            json.dump(result, fh, indent=1)


if __name__ == "__main__":
    main()
