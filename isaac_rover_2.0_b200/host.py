"""Host-buffer front end of the hot path: the call a simulator that keeps its state in HOST memory makes.

`submit()` enqueues one env step: pinned host -> device copies of this step's poses / joints / actions, the device hot path
(RoverTask.hot_step, two library calls), and -- on a second stream -- device -> pinned host copies of obs_buf / rew_buf /
reset_buf.  `result(slot)` waits for that step's copies and returns the host tensors.  Two slots (double buffering): the
28.7 MB observation read-back of step i overlaps the kernels of step i+1, and the inputs of step i+1 are uploaded on a third
stream into the other slot's device buffers while step i still computes (measured: small uploads queued on the compute stream
start together with the previous step's read-back and wait behind it, +0.2 ms per step).  `step()` = submit + result (no overlap).
bench.py's `e2e` number times submit/result in a loop where every step's inputs are copied in and every step's results are
read on the host.

`packed_obs=True`: the heightmap observation columns are produced and read back as the fp16 values they are by construction
(obs = fp16(dist / 2) widened to f32, rover.py:324-325), i.e. lossless at half the bytes: result() then returns
(obs_proprio f32 [N,4], obs_heightmap f16 [N,1746], rew, reset); `obs_f32(slot)` widens them on the host when a caller wants
the reference's [N,1750] f32 layout.  With 8 GPUs reading 28.7 MB each per step the host link is the bottleneck; this halves it.
"""
import torch


class HostPipeline:
    def __init__(self, task, depth=2, packed_obs=False, device_reset=False):
        self.task = task
        self.depth = depth
        self.packed_obs = packed_obs
        # device_reset: every step starts with the reset half of pre_physics_step on the device (RoverTask.hot_step); the mask it
        # consumes is the PREVIOUS step's reset_buf, which lives in the previous slot's buffer (read only: it may be in flight to
        # the host)
        self.device_reset = device_reset
        self._prev_reset = None
        N, dev = task.num_envs, torch.device(task._device)
        self.dev = dev
        pin = dict(pin_memory=True)
        mk = lambda shape, dt: [torch.empty(shape, dtype=dt, **pin) for _ in range(depth)]      # noqa: E731
        self.h_pos, self.h_quat = mk((N, 3), torch.float32), mk((N, 4), torch.float32)
        self.h_joints, self.h_actions = mk((N, 13), torch.float32), mk((N, 2), torch.float32)
        self.h_obs, self.h_rew, self.h_reset = mk((N, task.num_observations), torch.float32), mk((N,), torch.float32), mk((N,), torch.int64)
        dk = lambda shape: [torch.empty(shape, dtype=torch.float32, device=dev) for _ in range(depth)]      # noqa: E731
        self.d_pos, self.d_quat, self.d_joints, self.d_actions = dk((N, 3)), dk((N, 4)), dk((N, 13)), dk((N, 2))
        self.d_obs = [torch.zeros((N, task.num_observations), dtype=torch.float32, device=dev) for _ in range(depth)]
        self.d_rew = [torch.zeros((N,), dtype=torch.float32, device=dev) for _ in range(depth)]
        self.d_reset = [torch.zeros((N,), dtype=torch.int64, device=dev) for _ in range(depth)]
        if packed_obs:
            n_hm = task.num_observations - 4
            self.d_obs16 = [torch.zeros((N, n_hm), dtype=torch.float16, device=dev) for _ in range(depth)]
            self.d_prop = [torch.zeros((N, 4), dtype=torch.float32, device=dev) for _ in range(depth)]
            self.h_obs16 = mk((N, n_hm), torch.float16)
            self.h_prop = mk((N, 4), torch.float32)
        self.copy_stream = torch.cuda.Stream(dev)
        self.up_stream = torch.cuda.Stream(dev)
        self.uploaded = [torch.cuda.Event() for _ in range(depth)]
        self.computed = [torch.cuda.Event() for _ in range(depth)]
        self.done = [None] * depth
        self.i = 0
        view = task._rover
        view.pos, view.quat, view.joints = self.d_pos[0], self.d_quat[0], self.d_joints[0]
        self.h2d_bytes = sum(t[0].numel() * t[0].element_size() for t in (self.h_pos, self.h_quat, self.h_joints, self.h_actions))
        outs = (self.h_obs16, self.h_prop, self.h_rew, self.h_reset) if packed_obs else (self.h_obs, self.h_rew, self.h_reset)
        self.d2h_bytes = sum(t[0].numel() * t[0].element_size() for t in outs)

    def submit(self, pos, quat, joints, actions):
        """pos/quat/joints/actions: host tensors (any memory).  Enqueues the step and returns its slot."""
        k = self.i % self.depth
        self.i += 1
        if self.done[k] is not None:
            self.done[k].synchronize()          # slot k's previous read-back (and so its staging copies) has finished
        cur = torch.cuda.current_stream(self.dev)
        # slot k's device inputs were last read by the step whose read-back has just been waited for
        with torch.cuda.stream(self.up_stream):
            for src, stage, dst in ((pos, self.h_pos[k], self.d_pos[k]), (quat, self.h_quat[k], self.d_quat[k]),
                                    (joints, self.h_joints[k], self.d_joints[k]), (actions, self.h_actions[k], self.d_actions[k])):
                if src.data_ptr() != stage.data_ptr():
                    stage.copy_(src)
                dst.copy_(stage, non_blocking=True)
            self.uploaded[k].record(self.up_stream)
        cur.wait_event(self.uploaded[k])
        t = self.task
        view = t._rover
        view.pos, view.quat, view.joints = self.d_pos[k], self.d_quat[k], self.d_joints[k]
        t.obs_buf, t.rew_buf, t.reset_buf = self.d_obs[k], self.d_rew[k], self.d_reset[k]
        t.obs16_buf = self.d_obs16[k] if self.packed_obs else None
        t.hot_step(self.d_actions[k], device_reset=self.device_reset and self._prev_reset is not None, reset_mask=self._prev_reset)
        self._prev_reset = self.d_reset[k]
        if self.packed_obs:
            self.d_prop[k].copy_(self.d_obs[k][:, :4])          # 64 KB, contiguous for the read-back
        self.computed[k].record(cur)
        self.copy_stream.wait_event(self.computed[k])
        with torch.cuda.stream(self.copy_stream):
            if self.packed_obs:
                self.h_obs16[k].copy_(self.d_obs16[k], non_blocking=True)
                self.h_prop[k].copy_(self.d_prop[k], non_blocking=True)
            else:
                self.h_obs[k].copy_(self.d_obs[k], non_blocking=True)
            self.h_rew[k].copy_(self.d_rew[k], non_blocking=True)
            self.h_reset[k].copy_(self.d_reset[k], non_blocking=True)
            ev = torch.cuda.Event()
            ev.record(self.copy_stream)
        self.done[k] = ev
        # the next step's kernels write d_obs[k'] of ANOTHER slot; slot k is rewritten only after done[k] (see above)
        return k

    def result(self, k):
        self.done[k].synchronize()
        if self.packed_obs:
            return self.h_prop[k], self.h_obs16[k], self.h_rew[k], self.h_reset[k]
        return self.h_obs[k], self.h_rew[k], self.h_reset[k]

    def obs_f32(self, k):
        """The reference's [N, 4+sparse+dense] f32 observation of slot k, assembled on the host (packed mode)."""
        self.done[k].synchronize()
        if not self.packed_obs:
            return self.h_obs[k]
        return torch.cat((self.h_prop[k], self.h_obs16[k].float()), 1)

    def close(self):
        """Wait for the copies in flight and drop the buffers (pinned host memory is returned to torch's caching allocator)."""
        for ev in self.done:
            if ev is not None:
                ev.synchronize()
        for name in ("h_obs", "h_obs16", "h_prop", "d_obs", "d_obs16", "d_prop", "h_rew", "h_reset", "d_rew", "d_reset"):
            if hasattr(self, name):
                setattr(self, name, None)
        self._prev_reset = None

    def step(self, pos, quat, joints, actions):
        """Synchronous convenience: returns pinned host (obs, rew, reset) of this step."""
        return self.result(self.submit(pos, quat, joints, actions))
