"""Observation hooks and the teacher-data recorder (SURVEY.md 8f-4): the per-step epilogues of
RoverTask.get_observations the reference's authors toggled by hand (rover.py:298-317 recorder, :326-329 noise / dropout /
offset / remove_idx masking).  One kernel each behind the C ABI (csrc/hooks.cu); no CPU path."""
import math

import torch

from . import _lib, model


class ObsHooks:
    """The four commented-out lines of rover.py:326-329 as switches.  Reference values: noise_std = 0.20 ** 0.5,
    dropout_p = 0.1, offset = 0.02, remove_idx = torch.load('remove_idx.pt') (rover.py:88; indices into obs[:, 4:])."""

    def __init__(self, num_observations, noise_std=0.0, dropout_p=0.0, offset=0.0, remove_idx=None, num_proprioceptive=4, seed=42,
                 device="cuda:0"):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("rover_b200: ObsHooks needs a CUDA device (there is no CPU path)")
        if not (0.0 <= dropout_p < 1.0) or noise_std < 0:
            raise ValueError("dropout_p must be in [0, 1) and noise_std >= 0")
        self.num_observations = int(num_observations)
        self.col0 = int(num_proprioceptive)
        self.noise_std, self.dropout_p, self.offset, self.seed = float(noise_std), float(dropout_p), float(offset), int(seed)
        self.mask = None
        if remove_idx is not None:
            idx = torch.as_tensor(remove_idx, dtype=torch.long).flatten() + self.col0          # rover.py:329
            if idx.numel() and (idx.min() < 0 or idx.max() >= self.num_observations):
                raise IndexError("remove_idx out of range")
            m = torch.zeros(self.num_observations, dtype=torch.uint8)
            m[idx] = 1
            self.mask = m.to(self.device)
        self._lib = _lib.load()

    @classmethod
    def reference_values(cls, num_observations, remove_idx=None, **kw):
        return cls(num_observations, noise_std=math.sqrt(0.20), dropout_p=0.1, offset=0.02, remove_idx=remove_idx, **kw)

    def apply(self, obs, epoch, env_offset=0):
        """In place on obs f32 [N, >= num_observations]; `epoch` = the step counter (a new draw per step)."""
        _lib.require_cuda(obs)
        if obs.dtype != torch.float32 or obs.dim() != 2 or obs.stride(1) != 1 or obs.shape[1] < self.num_observations:
            raise RuntimeError("obs must be float32 [N, >=%d] with unit column stride" % self.num_observations)
        with torch.cuda.device(obs.device):
            _lib.check(self._lib.rvb_obs_hooks(_lib.ptr(obs), obs.stride(0), obs.shape[0], self.num_observations, self.col0,
                                               self.noise_std, self.dropout_p, self.offset, _lib.ptr(self.mask), self.seed,
                                               int(epoch), int(env_offset), _lib.stream_of(obs)))
        return obs


class TeacherRecorder:
    """rover.py:174-180,298-317: a [T, N, 1 + num_actions + num_observations] block filled one step per call and written to
    `teacher_dataset_<nr>.pt` in the reference's dict layout when full.  The block lives on the device (the reference keeps
    it in host memory and pays a device-to-host copy of obs_buf per step).

    `obs` is obs_buf (f32 [N, >= num_observations]) or the fused step's packed observation `(obs_buf[:, :p], obs16_buf)`
    (proprio f32 [N, >=p], heightmap f16 [N, >= num_observations - p]; rvb_teacher_record_packed), which the kernel widens into
    the same f32 row.  RoverTask hands the recorder the packed pair whenever obs16_buf is set.

    packed=False: the block is `teacher_dataset`, f32 [T, N, 3 + num_observations], one row [reset_info, a0, a1, obs] per env.
    packed=True: the block keeps the heightmap columns as the fp16 values they are (half the device memory: 3520 instead of
    7012 bytes per env-step with the shipped 1750 columns) in two parts:
      teacher_head       f32 [T, N, 3 + p]  the first 3 + p columns of every row: reset_info, a0, a1, the proprioceptive columns;
      teacher_heightmap  f16 [T, N, num_observations - p]  the heightmap columns.
    `widened_step(t)` gives timestep t's f32 rows [N, 3 + num_observations].  Such a recorder takes the packed pair only.  Either
    way the file holds the reference's f32 block, widened on the device one timestep at a time."""

    def __init__(self, num_envs, num_observations, num_sparse, num_dense, num_proprioceptive=4, steps=5 * 30, device="cuda:0",
                 directory=".", save=True, packed=False):
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise RuntimeError("rover_b200: TeacherRecorder needs a CUDA device (there is no CPU path)")
        self.num_envs, self.num_observations = int(num_envs), int(num_observations)
        self.num_proprioceptive = int(num_proprioceptive)
        if not 0 <= self.num_proprioceptive < self.num_observations:
            raise ValueError("num_proprioceptive must be in [0, num_observations)")
        self.packed = bool(packed)
        self.info = {"reset": 1, "actions": 2, "proprioceptive": num_proprioceptive, "sparse": num_sparse, "dense": num_dense}
        if self.packed:
            self.teacher_head = torch.empty((steps, num_envs, 3 + self.num_proprioceptive), device=self.device)
            self.teacher_heightmap = torch.empty((steps, num_envs, self.num_observations - self.num_proprioceptive),
                                                 device=self.device, dtype=torch.float16)
        else:
            self.teacher_dataset = torch.empty((steps, num_envs, 3 + num_observations), device=self.device)     # rover.py:178
        self.curr_timestep = 0
        self.dataset_nr = 0
        self.directory, self.save = directory, save
        self.last_file = None
        self._lib = _lib.load()

    def _observation(self, obs):
        """obs checked: the f32 rows, or the packed pair (proprio, heightmap).  Raises before anything touches a device."""
        p, e = self.num_proprioceptive, self.num_observations - self.num_proprioceptive
        if isinstance(obs, tuple):
            proprio, heightmap = model.packed_obs(obs, p, e, what="obs")
            if proprio.shape[0] != self.num_envs:
                raise RuntimeError("packed obs must have %d rows" % self.num_envs)
            return proprio, heightmap
        if self.packed:
            raise RuntimeError("TeacherRecorder(packed=True) records the packed observation (proprio float32 [N, >=%d], heightmap "
                               "float16 [N, >=%d]) only, not float32 rows: the heightmap columns of float32 rows need not be fp16 "
                               "values (after the observation hooks' noise, dropout or offset they are not), so the fp16 block "
                               "would change them; record float32 rows with packed=False" % (p, e))
        if (not isinstance(obs, torch.Tensor) or obs.dtype != torch.float32 or obs.dim() != 2 or obs.stride(1) != 1
                or obs.shape[0] != self.num_envs or obs.shape[1] < self.num_observations):
            raise RuntimeError("obs must be float32 [%d, >=%d] or the packed pair (proprio float32 [%d, >=%d], heightmap float16 "
                               "[%d, >=%d])" % (self.num_envs, self.num_observations, self.num_envs, p, self.num_envs, e))
        return obs, None

    def record(self, reset_info, actions, obs):
        """One step: row = [reset_info, actions, obs] per env (rover.py:299-300,364,374-375).  Returns the path of the file
        written when this call filled the block, else None."""
        obs, heightmap = self._observation(obs)
        _lib.require_cuda(reset_info, actions, obs, heightmap)
        reset_info = reset_info.to(torch.float32).contiguous()
        actions = actions.to(torch.float32)
        if actions.stride(1) != 1:
            actions = actions.contiguous()
        t = self.curr_timestep
        with torch.cuda.device(obs.device):
            if heightmap is None:
                row = self.teacher_dataset[t]
                _lib.check(self._lib.rvb_teacher_record(_lib.ptr(reset_info), _lib.ptr(actions), actions.stride(0), _lib.ptr(obs),
                                                        obs.stride(0), self.num_envs, self.num_observations, _lib.ptr(row),
                                                        row.stride(0), _lib.stream_of(obs)))
            elif self.packed:
                self._record_packed(reset_info, actions, obs, heightmap, self.teacher_head[t], self.teacher_heightmap[t])
            else:
                self._record_packed(reset_info, actions, obs, heightmap, self.teacher_dataset[t], None)
        self.curr_timestep += 1
        if self.curr_timestep < (self.teacher_head if self.packed else self.teacher_dataset).shape[0]:
            return None
        self.curr_timestep = 0                                                    # rover.py:302-317
        path = None
        if self.save:
            import os
            path = os.path.join(self.directory, "teacher_dataset_" + str(self.dataset_nr) + ".pt")
            torch.save({"info": dict(self.info), "data": self._host_block()}, path)
        self.last_file = path
        self.dataset_nr += 1
        if self.packed:
            self.teacher_head = torch.empty_like(self.teacher_head)
            self.teacher_heightmap = torch.empty_like(self.teacher_heightmap)
        else:
            self.teacher_dataset = torch.empty_like(self.teacher_dataset)
        return path

    def _record_packed(self, reset_info, actions, proprio, heightmap, rec, rec16):
        """rvb_teacher_record_packed: widened into the f32 row block `rec` (rec16 None), or split into `rec` + `rec16`."""
        _lib.check(self._lib.rvb_teacher_record_packed(
            _lib.ptr(reset_info), _lib.ptr(actions), model._row_stride(actions), _lib.ptr(proprio), model._row_stride(proprio),
            self.num_proprioceptive, _lib.ptr(heightmap), model._row_stride(heightmap), self.num_observations - self.num_proprioceptive,
            self.num_envs, _lib.ptr(rec), model._row_stride(rec), _lib.ptr(rec16), 0 if rec16 is None else model._row_stride(rec16),
            _lib.stream_of(proprio)))

    def widened_step(self, t, out=None):
        """Timestep t of a packed block as the f32 rows [N, 3 + num_observations] of the reference's layout, widened on the device
        (into `out` when given)."""
        if not self.packed:
            raise RuntimeError("widened_step: the recorder keeps f32 rows already (teacher_dataset)")
        head, hm = self.teacher_head[t], self.teacher_heightmap[t]
        if out is None:
            out = torch.empty((self.num_envs, 3 + self.num_observations), device=head.device)
        p = self.num_proprioceptive
        with torch.cuda.device(head.device):
            self._record_packed(head[:, 0].contiguous(), head[:, 1:3], head[:, 3:3 + p], hm, out, None)
        return out

    def _host_block(self):
        """The block as the reference's f32 [T, N, 3 + num_observations] host tensor; a packed block is widened one timestep at a
        time on the device and copied down, so no fp16 value is converted on the host."""
        if not self.packed:
            return self.teacher_dataset.cpu()
        steps = self.teacher_head.shape[0]
        data = torch.empty((steps, self.num_envs, 3 + self.num_observations), dtype=torch.float32)
        rows = None
        for t in range(steps):
            rows = self.widened_step(t, rows)
            data[t].copy_(rows)
        return data
