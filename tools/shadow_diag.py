"""GPU diagnostic: production (shadow) ray-cast vs the tiled and per-pair kernels on the benchmark world; prints
mismatch statistics and per-variant timings.  python tools/shadow_diag.py [N]"""
import os
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import isaac_rover_b200 as R      # noqa: E402

N = int(sys.argv[1]) if len(sys.argv) > 1 else 4096


def timed(fn, reps=30, warm=3):
    """median / min of per-launch CUDA-event times [ms]"""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in ev:
        a.record()
        fn()
        b.record()
    torch.cuda.synchronize()
    t = sorted(a.elapsed_time(b) for a, b in ev)
    return t[len(t) // 2], t[0]
w = R.synth.make_world(length=200.0, nv=708, K=200, n_stones=2000, seed=42, build_index=None)
t0 = time.perf_counter()
w.map_indices = R.build_knn_index(w.triangles, w.vertices, w.G, w.res, w.K, device="cuda:0")
torch.cuda.synchronize()
print("index build %.2f s" % (time.perf_counter() - t0))
t0 = time.perf_counter()
cam = R.Camera("cuda:0", torch.tensor([0, 0, 0.0]), assets=(w.map_indices, w.triangles, w.vertices))
torch.cuda.synchronize()
print("layer create %.2f s, %.2f GB" % (time.perf_counter() - t0, cam.layer.bytes() / 1e9))
st = {k: v.cuda() for k, v in R.synth.make_env_state(w, N, seed=100).items()}
eul = R.tensor_quat_to_eul(st["quat"])
out = {}
for v in (3, 0, 2):
    cam.variant = v
    for _ in range(2):
        d, pt, s = cam.get_depths(st["pos"], eul, want_hits=True, want_pt=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        d, pt, s = cam.get_depths(st["pos"], eul, want_hits=False, want_pt=False)
    e1.record()
    torch.cuda.synchronize()
    print("variant %d: %.3f ms per launch (%d envs)" % (v, e0.elapsed_time(e1) / 5, N))
    d, pt, s = cam.get_depths(st["pos"], eul, want_hits=True, want_pt=False)
    out[v] = (d.clone(), cam.last_hit_slot.clone(), cam.last_hit_tri.clone())
import os as _os
cam.variant = 0
med, mn = timed(lambda: cam.get_depths(st["pos"], eul, want_pt=False))
d, _, _ = cam.get_depths(st["pos"], eul, want_pt=False)
print("shadow: median %.3f ms, min %.3f ms, equal to variant 3: %s" % (med, mn, bool(torch.equal(d.view(torch.int16), out[3][0].view(torch.int16)))))
for ns in ("0", "444", "0", "444"):
    _os.environ["RVB_SHADOW_SPLIT"] = ns
    cam.variant = 0
    med, mn = timed(lambda: cam.get_depths(st["pos"], eul, want_pt=False), reps=30)
    d, _, _ = cam.get_depths(st["pos"], eul, want_pt=False)
    print("split envs %s: median %.3f ms, min %.3f, equal to variant 3: %s" % (ns, med, mn, bool(torch.equal(d.view(torch.int16), out[3][0].view(torch.int16)))))
_os.environ.pop("RVB_SHADOW_SPLIT")
for msh in ("1", "0", "1", "0"):
    _os.environ["RVB_SHADOW_SH"] = msh
    cam.variant = 0
    med, mn = timed(lambda: cam.get_depths(st["pos"], eul, want_pt=False), reps=30)
    d, _, _ = cam.get_depths(st["pos"], eul, want_pt=False)
    print("min bin shift %s: median %.3f ms, min %.3f, equal to variant 3: %s" % (msh, med, mn, bool(torch.equal(d.view(torch.int16), out[3][0].view(torch.int16)))))
_os.environ.pop("RVB_SHADOW_SH")
for trn in ("8", "12", "16", "8", "16"):
    _os.environ["RVB_SHADOW_TASK_RAYS"] = trn
    cam.variant = 0
    med, mn = timed(lambda: cam.get_depths(st["pos"], eul, want_pt=False), reps=30)
    d, _, _ = cam.get_depths(st["pos"], eul, want_pt=False)
    print("rays per task %s: median %.3f ms, min %.3f, equal to variant 3: %s" % (trn, med, mn, bool(torch.equal(d.view(torch.int16), out[3][0].view(torch.int16)))))
_os.environ.pop("RVB_SHADOW_TASK_RAYS")
for cs in ("0.7", "0.9"):
    _os.environ["RVB_COS_STEEP"] = cs
    cam.variant = 0
    med, mn = timed(lambda: cam.get_depths(st["pos"], eul, want_pt=False), reps=15)
    d, _, _ = cam.get_depths(st["pos"], eul, want_pt=False)
    print("cos_steep %s: median %.3f ms, min %.3f, equal to variant 3: %s" % (cs, med, mn, bool(torch.equal(d.view(torch.int16), out[3][0].view(torch.int16)))))
_os.environ.pop("RVB_COS_STEEP")

# the same without the 1 % strongly tilted envs
st2 = dict(st)
eul2 = eul.clone()
eul2[:, :2] = eul2[:, :2].clamp(-0.25, 0.25)
for v in (3, 0):
    cam.variant = v
    med, mn = timed(lambda: cam.get_depths(st["pos"], eul2, want_pt=False), reps=15)
    print("no tilted envs, variant %d: median %.3f ms, min %.3f" % (v, med, mn))
ref = out[3]
for v in (0, 2):
    neq = out[v][0].view(torch.int16) != ref[0].view(torch.int16)
    nslot = out[v][1] != ref[1]
    print("variant %d vs 3: %d / %d distances differ (%d envs), %d slots differ" % (
        v, int(neq.sum()), neq.numel(), int(neq.any(1).sum()), int(nslot.sum())))
    if neq.any():
        idx = neq.nonzero()[:10]
        for e, p in idx.tolist():
            print("   env %d ray %d: got %s (slot %d tri %d) want %s (slot %d tri %d)  roll/pitch %.2f %.2f pos %s" % (
                e, p, out[v][0][e, p].item(), out[v][1][e, p].item(), out[v][2][e, p].item(), ref[0][e, p].item(),
                ref[1][e, p].item(), ref[2][e, p].item(), eul[e, 0].item(), eul[e, 1].item(), st["pos"][e].tolist()))
        miss_not_hit = (neq & (out[v][0] == 11)).sum().item()
        print("   of those, %d are misses where the reference kernel hits" % miss_not_hit)

sys.stdout.flush()
os.environ["RVB_SHADOW_DBG"] = "1"
cam.variant = 0
cam.get_depths(st["pos"], eul, want_pt=False)
torch.cuda.synchronize()
os.environ.pop("RVB_SHADOW_DBG")
