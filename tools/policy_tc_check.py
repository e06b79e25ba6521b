"""GPU check of the tensor-core policy path (variant 2) against the FFMA path (variant 1) + timings."""
import os, sys, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import isaac_rover_b200 as R
lib = R._lib.load()
torch.manual_seed(1)
net = R.model.NetworkInfo([256, 160, 128], [80, 60], [80, 60], [80, 60], "leakyrelu")
info = R.model.ObserverationInfo(4, 634, 1112, 0)
actor = R.model.StochasticActorHeightmap(1750, 2, net, info, device="cuda:0")
critic = R.model.DeterministicHeightmap(1750, 2, net, info, device="cuda:0")
for N in (128, 1000, 4096, 131072):
    obs = torch.rand(N, 1750, device="cuda")
    obs[:, 4:] = (obs[:, 4:] * 5.5).half().float()
    out = {}
    for v in (1, 2):
        lib.rvb_policy_variant(v)
        m, c = R.model.compute_pair(actor, critic, obs)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(3):
            R.model.compute_pair(actor, critic, obs)
        e0.record()
        for _ in range(10):
            R.model.compute_pair(actor, critic, obs)
        e1.record()
        torch.cuda.synchronize()
        out[v] = (m.clone(), c.clone(), e0.elapsed_time(e1) / 10)
    print("N %6d: variant 1 %.4f ms, variant 2 (tcgen05 first layers) %.4f ms; max |diff| mean %.2e value %.2e" % (
        N, out[1][2], out[2][2], (out[1][0] - out[2][0]).abs().max().item(), (out[1][1] - out[2][1]).abs().max().item()), flush=True)
lib.rvb_policy_variant(2)
