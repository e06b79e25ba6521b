"""`RoverTask` hot path -- mirror of tasks/rover.py (RoverTask :80-676, Memory :60-77) and of the buffer
contract of tasks/base/rl_task.py (:98-107 buffers, :239-259 post_physics_step ordering).

Only the per-step data-parallel path is here; Isaac Sim scene set-up, PhysX stepping, reset poses, skrl
and the teacher/student policies stay where they are (SURVEY.md section 8).  The simulator is whatever object is
passed as `rover_view`: it must offer the four ArticulationView calls the reference makes on this path
  get_world_poses() -> (pos f32 [N,3], quat_wxyz f32 [N,4]),  get_joint_positions() -> f32 [N,13],
  set_joint_position_targets(pos [N,4], indices=None, joint_indices=...),
  set_joint_velocity_targets(vel [N,6], indices=None, joint_indices=...)           (rover.py:274-275,291,412-414)
State lives in the same attribute names as the reference (obs_buf, rew_buf, reset_buf, progress_buf, extras,
target_positions, initial_pos, stone_info, linear_velocity, angular_velocity, rover_positions, rover_rotation,
rover_rot, heading_diff, rock_collison, curriculum_level, rew_scales, max_episode_length).
"""
import ctypes as C
import math

import torch

from . import _lib
from .camera import Camera
from .kinematics import Ackermann
from .rock_detect import Rock_Detection
from .tensor_quat_to_euler import tensor_quat_to_eul

DEFAULT_REWARDS = dict(pos_reward=1.0, terminalReward=0, collision_reward=0.3, heading_contraint_reward=0.05,
                       motion_contraint_reward=-0.01, goal_angle_reward=0.3, boogie_contraint_reward=0.5)   # Rover.yaml:37-46

STAT_NAMES = ("envs", "reward_sum", "pos_reward_sum", "collisions", "uprightness_sum", "heading_penalty_sum",
              "motion_penalty_sum", "goal_angle_penalty_sum", "resets", "timeouts", "tilt_resets", "too_far_resets",
              "goals_reached", "collision_resets", "target_dist_sum", "reserved")


def _f32(t):
    """t as a contiguous f32 tensor (itself when it already is one)."""
    return t if (t.dtype == torch.float32 and t.is_contiguous()) else t.to(torch.float32).contiguous()


class Memory():
    """[num_envs, num_states, horizon] shift register, newest at index 0 (rover.py:60-77).  The shift is done
    in place by rvb_history_push instead of cat + slice re-allocation."""

    def __init__(self, num_envs, num_states, horizon, device) -> None:
        self.tracker = torch.zeros((num_envs, num_states, horizon), device=device)
        self.device = device
        self.num_envs = num_envs
        self.num_states = num_states
        self.horizon = horizon

    def get_state(self, timestep):
        data = self.tracker[:, :, timestep]
        if data.shape[1] == 1:
            return data.squeeze(1)
        return data

    def input_state(self, state):
        _lib.require_cuda(self.tracker, state)
        lib = _lib.load()
        st = state.to(torch.float32)
        if st.dim() != 1:
            st = st.reshape(-1)
        if st.shape[0] != self.num_envs * self.num_states:
            raise ValueError("Memory.input_state: expected %d values" % (self.num_envs * self.num_states))
        stride = st.stride(0) if st.shape[0] > 1 else 1
        with torch.cuda.device(self.tracker.device):
            _lib.check(lib.rvb_history_push(_lib.ptr(self.tracker), self.num_envs * self.num_states, self.horizon,
                                            _lib.ptr(st), stride, _lib.stream_of(self.tracker)))


class RoverTask():
    def __init__(self, rover_view, num_envs, terrain_assets, rock_assets, stone_info, heightmap,
                 device='cuda:0', shift=None, rewards=None, horizontal_scale=0.025, vertical_scale=1,
                 sem=_lib.SEM_TORCH_CUDA, num_envs_total=None, rover_name="rover_view", compact_terrain=False):
        """terrain_assets / rock_assets: (map_indices [K,G,G], triangles, vertices) of knn_terrain / knn_rocks
        (None -> loaded from the reference's relative paths); stone_info f32 [S,7] (read_stone_info);
        heightmap f32 [H,H] (heightmap_tensor.pt, rover.py:210).
        compact_terrain: the heightmap layer gives back its copy of the index (Camera(compact=True)): same step, 3.2 GB less."""
        self._lib = _lib.load()
        self._device = device
        self._rover = rover_view
        self._rover_name = getattr(rover_view, "name", rover_name)
        self._num_envs = self.num_envs = num_envs
        self.num_envs_total = num_envs if num_envs_total is None else num_envs_total
        self.sem = sem
        self.shift = torch.tensor([0, 0, 0.0], device=device) if shift is None else shift.to(device)
        self.Camera = Camera(device, self.shift, debug=False, assets=terrain_assets, sem=sem, compact=compact_terrain)
        self.num_exteroceptive = self.Camera.get_num_exteroceptive()
        self.Rock_detector = Rock_Detection(device, self.shift, debug=False, assets=rock_assets, sem=sem)
        self.global_step = 0
        self._num_proprioceptive = 4
        self._num_observations = self.num_observations = (
            self._num_proprioceptive + self.Camera.heightmap.get_num_sparse_vector()
            + self.Camera.heightmap.get_num_dense_vector())
        self._num_actions = self.num_actions = 2
        self.curriculum_level = 1                                   # rover.py:104 (raised to 2 at :353)
        self.max_episode_length = 3000                              # rover.py:119
        self.is_evaluation = False
        self.save_teacher_data = False                              # rover.py:151; set a hooks.TeacherRecorder in `teacher_recorder`
        self.teacher_recorder = None
        self.reset_info = torch.zeros(num_envs, device=device)      # rover.py:180
        self._teacher_actions = torch.zeros((num_envs, 2), device=device)
        self.obs_hooks = None                                       # hooks.ObsHooks: rover.py:326-329 when enabled
        self.target_positions = torch.zeros((num_envs, 3), device=device, dtype=torch.float32)
        self.initial_pos = torch.zeros((num_envs, 3), device=device, dtype=torch.float32)
        self.stone_info = stone_info.to(device).float().contiguous()
        self.heightmap = heightmap.to(device).float().contiguous() if heightmap is not None else None
        self.horizontal_scale = horizontal_scale                    # rover.py:212
        self.vertical_scale = vertical_scale
        self.linear_velocity = Memory(num_envs, 1, 3, device)       # rover.py:154-155
        self.angular_velocity = Memory(num_envs, 1, 3, device)
        self.rew_scales = dict(DEFAULT_REWARDS if rewards is None else rewards)
        # RLTask.cleanup buffers (rl_task.py:98-107)
        self.obs_buf = torch.zeros((num_envs, self._num_observations), device=device, dtype=torch.float)
        self.rew_buf = torch.zeros(num_envs, device=device, dtype=torch.float)
        self.reset_buf = torch.ones(num_envs, device=device, dtype=torch.long)
        self.progress_buf = torch.zeros(num_envs, device=device, dtype=torch.long)
        self.states_buf = torch.zeros((num_envs, 0), device=device, dtype=torch.float)
        self.extras = {}
        self.rover_positions = None
        self.rover_rotation = None
        self.rover_rot = None
        self.heading_diff = torch.zeros(num_envs, device=device)
        self.rock_collison = torch.zeros(num_envs, device=device, dtype=torch.long)
        self.rock_wheel_dist = None
        self.rock_body_dist = None
        # episode statistics (per-rank sums; all-reduced by dist.reduce_stats)
        self.stats = torch.zeros(_lib.N_STATS, device=device, dtype=torch.float64)
        self._stats_scratch = torch.zeros(int(self._lib.rvb_stats_scratch_len(num_envs)), device=device,
                                          dtype=torch.float64)
        self._ex = dict(pos_reward=torch.zeros(num_envs, device=device),
                        collision_penalty=torch.zeros(num_envs, device=device, dtype=torch.long),
                        uprightness_penalty=torch.zeros(num_envs, device=device),
                        heading_contraint_penalty=torch.zeros(num_envs, device=device),
                        motion_contraint_penalty=torch.zeros(num_envs, device=device),
                        goal_angle_penalty=torch.zeros(num_envs, device=device))
        self._count = torch.zeros(1, device=device, dtype=torch.int32)
        # optional packed observation of the fused step: f16 [N, sparse+dense]; when set, obs_buf[:, 4:] is not written
        self.obs16_buf = None
        # parity-test hooks (unfused path only): f32 [N,6] sin/cos of -roll,-pitch,-yaw and f32 [N,18] sin/cos of joints 0..8
        # to use instead of the device's sinf/cosf, so that tests can demand bit-identical rays (libm differs in the last ulp)
        self.parity_trig = None
        self.parity_joint_trig = None
        self._shift_host = None
        self.reset_seed = 42                                        # cfg/config.yaml:11
        self.env_offset = 0                                         # global id of local env 0 (env shards, dist.env_shard)
        self.reset_counters = torch.zeros(3, device=device, dtype=torch.int32)      # envs reset, goals drawn, envs out of attempts
        self._reset_next = None
        self._fused = None
        self.joint_position_targets = None
        self.joint_velocity_targets = None

    # ------------------------------------------------------------------ helpers
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(torch.device(self._device)).cuda_stream)

    # ------------------------------------------------------------------ drop-in constructor (rover.py:81-87)
    @classmethod
    def from_reference(cls, name, sim_config, env, offset=None, rover_view=None, stone_info=None, heightmap=None,
                       terrain_assets=None, rock_assets=None, **kw):
        """The reference's constructor signature `RoverTask(name, sim_config, env, offset)` (rover.py:81-87): numEnvs and the
        reward scales are read from `sim_config.task_config` the way rover.py:113,158 read them, the terrain / rock assets
        are loaded from the reference's relative paths (camera.py:154-161) unless given, `env` is kept for the
        `is_playing()` guard of post_physics_step (rl_task.py:250).  What Isaac Sim creates in set_up_scene -- the rover view,
        stone_info (rover.py:144) and the height grid (rover.py:210) -- is passed by keyword or attached afterwards
        (`task._rover = RoverView(...)`, `task.stone_info = ...`, `task.heightmap = ...`)."""
        cfg = getattr(sim_config, "task_config", None) or {}
        env_cfg = cfg.get("env", {}) if hasattr(cfg, "get") else {}
        n = int(env_cfg.get("numEnvs", kw.pop("num_envs", 1)))
        rewards = dict(DEFAULT_REWARDS)
        for k in DEFAULT_REWARDS:
            if k in (cfg.get("rewards", {}) if hasattr(cfg, "get") else {}):
                rewards[k] = cfg["rewards"][k]
        if stone_info is None:
            stone_info = torch.zeros((1, 7), dtype=torch.float32)
            stone_info[0, :2] = 1e9                         # one stone infinitely far away: every goal / spawn point is valid
        task = cls(rover_view, n, terrain_assets, rock_assets, stone_info, heightmap, rewards=rewards, **kw)
        task._name, task._sim_config, task._env, task._offset = name, sim_config, env, offset
        task._cfg = getattr(sim_config, "config", None)
        task._task_cfg = cfg
        return task

    # ------------------------------------------------------------------ RLTask.post_physics_step (rl_task.py:239-259)
    def get_states(self):
        """rl_task.py:210-216 (asymmetric-critic states buffer; the rover task has num_states = 0)."""
        return self.states_buf

    def get_extras(self):
        """rl_task.py:218-223: the rover task fills `extras` in calculate_metrics."""
        return self.extras

    def _is_playing(self):
        env = getattr(self, "_env", None)
        world = getattr(env, "_world", None)
        return True if world is None else bool(world.is_playing())

    def post_physics_step(self):
        self.progress_buf[:] += 1
        if self._is_playing():                                      # rl_task.py:250
            self.get_observations()
            self.get_states()
            self.calculate_metrics()
            self.is_done()
            self.get_extras()
        return self.obs_buf, self.rew_buf, self.reset_buf, self.extras

    def hot_step(self, actions, fused=True, device_reset=False, reset_mask=None):
        """One env-step of the hot path with PhysX excluded: the action half of pre_physics_step (history,
        Ackermann, joint targets; rover.py:343,366-414) followed by post_physics_step (rl_task.py:239-259).
        device_reset=True runs the reset half of pre_physics_step first (rover.py:356-361: book-keeping, goal
        re-sampling against stone_info, target heights) for every env whose reset_buf is set, on the device
        (rvb_reset_targets; pose resets stay with the simulator: `_rover.reset_idx_masked(mask, initial_pos)` when the
        view offers it).  fused=True enqueues the rest of the step with two library calls (rvb_env_pre + rvb_env_post) on
        the pose the view holds after the reset half; fused=False makes the reference's sequence of calls (same results,
        ~25 host round trips).  The observation hooks and the teacher recorder (rover.py:298-317,326-329) run on both paths.
        reset_mask: the mask to consume instead of reset_buf (i64 [N], read only -- used by HostPipeline, whose reset_buf
        rotates between slots)."""
        self.global_step += 1                                       # rover.py:341
        if fused:
            self._refuse_hooks_with_obs16("hot_step")
        if device_reset:
            self._reset_half(reset_mask=reset_mask)
        if not fused:
            _, quat = self._rover.get_world_poses()
            self.rover_rot = tensor_quat_to_eul(quat)
            self.apply_actions(actions)
            return self.post_physics_step()
        pos, quat, joints = self._view_state()
        self._action_half(actions, quat)
        out = self._observation_half(pos, quat, joints)
        self._hand_targets()
        return out

    # ------------------------------------------------------------------ the fused step split at the simulator's boundary
    def pre_physics_step_fused(self, actions, max_attempts=64) -> None:
        """pre_physics_step_device (rover.py:338-414, reset path on the device) for a loop in which the simulator steps between
        the halves: the action half is ONE launch (rvb_env_pre) instead of four, rover_rot is the euler of the pose the view holds
        now.  Same side effects as pre_physics_step_device."""
        self.global_step += 1
        self.rover_loc, quat = self._rover.get_world_poses()
        # The action half is enqueued BEFORE the reset half, so rover_rot is the pose before the simulator's pose reset, as
        # rover.py:343 takes it before :356.  Moving it ahead changes nothing else: the reset half writes goal targets, progress,
        # reset flags and reset_info, none of which the action half (histories, steering, wheel velocities) reads or writes.
        self._action_half(actions, _f32(quat))
        self._reset_half(max_attempts=max_attempts)
        self._hand_targets()                                        # after the resets, as apply_actions does

    def post_physics_step_fused(self):
        """post_physics_step (rl_task.py:239-259) after pre_physics_step_fused and the simulator's step: ONE library call
        (rvb_env_post) on the poses and joints the view holds now, is_done on the rover_rot of the pre half.  Honours obs16_buf
        like hot_step (then obs_buf[:, 4:] is not written, and the teacher recorder reads (obs_buf[:, :4], obs16_buf))."""
        if not self._is_playing():                                  # rl_task.py:241 comes before the guard at :250
            self.progress_buf[:] += 1
            return self.obs_buf, self.rew_buf, self.reset_buf, self.extras
        pos, quat, joints = self._view_state()
        self._refuse_hooks_with_obs16("post_physics_step_fused")
        if self.rover_rot is None:
            raise RuntimeError("post_physics_step_fused: no rover_rot; the pre-physics half has not run")
        return self._observation_half(pos, quat, joints)

    def _reset_half(self, reset_mask=None, max_attempts=64):
        """The reset half of pre_physics_step on the device (rover.py:356-361) for the envs set in reset_mask (default reset_buf):
        reset_info, the view's pose reset, then reset_targets_device."""
        mask = self.reset_buf if reset_mask is None else reset_mask
        # rover.py:420-422 without the host-side nonzero(): when any env resets, the reference sets reset_info of EVERY env
        if self.save_teacher_data:
            any_reset = (mask != 0).any().to(self.reset_info.dtype)
            torch.maximum(self.reset_info, any_reset.expand_as(self.reset_info), out=self.reset_info)
        if hasattr(self._rover, "reset_idx_masked"):
            self._rover.reset_idx_masked(mask.clone(), self.initial_pos)
        self.reset_targets_device(max_attempts=max_attempts, reset_mask=reset_mask)

    def _view_state(self):
        """The poses and joint positions the view holds now, as contiguous f32 device tensors."""
        pos, quat = self._rover.get_world_poses()
        joints = self._rover.get_joint_positions()
        pos, quat, joints = _f32(pos), _f32(quat), _f32(joints)
        _lib.require_cuda(pos, quat, joints)
        return pos, quat, joints

    def _action_half(self, actions, quat):
        """rvb_env_pre on `quat`: rover_rot, both histories and the joint targets, which _hand_targets gives to the view."""
        act = self._actions_f32(actions)
        _lib.require_cuda(quat, act)
        if self.save_teacher_data:                                  # rover.py:373-375
            self._teacher_actions = act[:, 0:2]
        fb = self._step_buffers()
        with torch.cuda.device(torch.device(self._device)):
            _lib.check(self._lib.rvb_env_pre(_lib.ptr(quat), _lib.ptr(act), self.num_envs, self.linear_velocity.horizon,
                                             _lib.ptr(self.linear_velocity.tracker), _lib.ptr(self.angular_velocity.tracker),
                                             _lib.ptr(fb["rot"]), _lib.ptr(fb["pos_t"]), _lib.ptr(fb["vel_t"]), self.sem,
                                             self._stream()))
        self.rover_rot = fb["rot"]

    def _observation_half(self, pos, quat, joints):
        """rvb_env_post on the view's state, is_done on rover_rot; the teacher recorder's row before it, the observation hooks
        (rover.py:326-329), attributes and extras after it."""
        fb = self._step_buffers()
        if self.save_teacher_data and self.teacher_recorder is not None:       # rover.py:298-317: BEFORE obs_buf is refreshed
            self.teacher_recorder.record(self.reset_info, self._teacher_actions, self._teacher_obs())
        want_rocks = self.curriculum_level >= 2
        io = self._step_io(pos, quat, joints, want_rocks)
        prm = self._params()
        cam = self.Camera
        with torch.cuda.device(torch.device(self._device)):
            _lib.check(self._lib.rvb_env_post(cam.layer.handle, self.Rock_detector.layer.handle if want_rocks else None,
                                              C.byref(prm), C.byref(io), _lib.ptr(self.rover_rot), _lib.ptr(cam.heightmap_distribution),
                                              self.num_exteroceptive, _lib.ptr(cam._col_a), _lib.ptr(cam._col_b), self.num_envs,
                                              self.linear_velocity.horizon, self._stream()))
        if not want_rocks:                                          # no rock kernel was launched
            _lib.launch_count -= 1
        if self.obs_hooks is not None:
            self.obs_hooks.apply(self.obs_buf, epoch=self.global_step, env_offset=self.env_offset)
        self.rover_positions, self.rover_rotation = pos, fb["euler"]
        self.rock_wheel_dist, self.rock_body_dist = (fb["wheel"], fb["body"]) if want_rocks else (None, None)
        self.extras.update(self._ex)
        self.extras["torque_penalty_driving"] = self.linear_velocity.tracker[:, 0, 0]      # rover.py:530-531
        self.extras["torque_penalty_steering"] = self.angular_velocity.tracker[:, 0, 0]
        return self.obs_buf, self.rew_buf, self.reset_buf, self.extras

    def _actions_f32(self, actions):
        dev = torch.device(self._device)
        ok = actions.dtype == torch.float32 and actions.is_contiguous() and actions.device == dev
        return actions if ok else actions.to(dev, torch.float32).contiguous()

    def _teacher_obs(self):
        """The observation the fused step's recorder row pairs with this step's actions: obs_buf, or with obs16_buf set the packed
        pair (obs_buf[:, :4], obs16_buf) -- the fused step then leaves obs_buf[:, 4:] unwritten.  The choice follows obs16_buf as it
        is now: a task that switches obs16_buf on or off between steps records, for the step after the switch, a buffer the previous
        step did not write."""
        if self.obs16_buf is None:
            return self.obs_buf
        return self.obs_buf[:, :self._num_proprioceptive], self.obs16_buf

    def _refuse_hooks_with_obs16(self, who):
        if self.obs_hooks is not None and self.obs16_buf is not None:
            raise RuntimeError("%s: observation hooks work on obs_buf (f32); they cannot be combined with the packed "
                               "fp16 observation output (obs16_buf)" % who)

    def _step_buffers(self):
        """Device outputs of the fused step and its halves that have no attribute of the reference's (allocated once)."""
        if self._fused is None:
            N, P, dev = self.num_envs, self.num_exteroceptive, torch.device(self._device)
            self._fused = dict(
                euler=torch.empty((N, 3), device=dev), dist=torch.empty((N, P), device=dev, dtype=torch.float16),
                wheel=torch.empty((N, 24), device=dev, dtype=torch.float16), body=torch.empty((N, 2), device=dev, dtype=torch.float16),
                pos_t=torch.empty((N, 4), device=dev), vel_t=torch.empty((N, 6), device=dev), rot=torch.empty((N, 3), device=dev))
        return self._fused

    def _step_io(self, pos, quat, joints, want_rocks):
        fb = self._fused
        e = self._ex
        return _lib.StepIO(*[_lib.ptr(t) for t in (pos, quat, joints, self.target_positions, self.linear_velocity.tracker,
                                                    self.angular_velocity.tracker, self.progress_buf, fb["euler"], self.heading_diff,
                                                    self.obs_buf)],
                           self.obs_buf.stride(0),
                           *[_lib.ptr(t) for t in (fb["dist"], fb["wheel"] if want_rocks else None, fb["body"] if want_rocks else None,
                                                    self.rock_collison if want_rocks else None, self.rew_buf, self.reset_buf,
                                                    e["pos_reward"], e["collision_penalty"], e["uprightness_penalty"],
                                                    e["heading_contraint_penalty"], e["motion_contraint_penalty"],
                                                    e["goal_angle_penalty"], self.stats, self._stats_scratch, self.obs16_buf)],
                           0 if self.obs16_buf is None else self.obs16_buf.stride(0))

    def _hand_targets(self):
        """rover.py:412-414: the joint targets of the action half go to the view."""
        pos_t, vel_t = self._fused["pos_t"], self._fused["vel_t"]
        self.joint_position_targets, self.joint_velocity_targets = pos_t, vel_t
        if hasattr(self._rover, "set_joint_position_targets"):
            self._rover.set_joint_position_targets(pos_t, indices=None, joint_indices=getattr(self._rover, "actuated_pos_indices", None))
            self._rover.set_joint_velocity_targets(vel_t, indices=None, joint_indices=getattr(self._rover, "actuated_vel_indices", None))

    # ------------------------------------------------------------------ get_observations (rover.py:272-336)
    def get_observations(self) -> dict:
        lib = self._lib
        if self.save_teacher_data and self.teacher_recorder is not None:       # rover.py:298-317: BEFORE obs_buf is refreshed --
            # the row pairs the actions of this step with the observation they were computed from
            self.teacher_recorder.record(self.reset_info, self._teacher_actions, self.obs_buf)
        pos, quat = self._rover.get_world_poses()
        self.rover_positions = pos.to(torch.float32).contiguous()
        self.rover_rotation = tensor_quat_to_eul(quat)
        lin_now = self.linear_velocity.tracker[:, 0, 0].contiguous()
        ang_now = self.angular_velocity.tracker[:, 0, 0].contiguous()
        with torch.cuda.device(torch.device(self._device)):
            _lib.check(lib.rvb_obs_proprio(_lib.ptr(self.rover_positions), _lib.ptr(self.rover_rotation),
                                           _lib.ptr(self.target_positions), _lib.ptr(lin_now), _lib.ptr(ang_now),
                                           self.num_envs, _lib.ptr(self.obs_buf), self.obs_buf.stride(0),
                                           _lib.ptr(self.heading_diff), self.sem, self._stream()))
        # heightmap: ray-cast with the sparse/dense gather + /2 fused into obs_buf[:, 4:] (rover.py:286-288,324-325)
        self.Camera.get_depths(self.rover_positions, self.rover_rotation, obs=self.obs_buf, want_pt=False, trig=self.parity_trig)
        # rock collision (rover.py:291-293)
        want = self.curriculum_level >= 2
        self.rock_wheel_dist, self.rock_body_dist = self.Rock_detector.get_collisions(
            self.rover_positions, self.rover_rotation, self._rover.get_joint_positions(), want_collision=want,
            trig=self.parity_trig, joint_trig=self.parity_joint_trig)
        if want:
            self.rock_collison = self.Rock_detector.last_collision
        if self.obs_hooks is not None:                              # rover.py:326-329
            self.obs_hooks.apply(self.obs_buf, epoch=self.global_step, env_offset=self.env_offset)
        return {self._rover_name: {"obs_buf": self.obs_buf}}

    def check_collision(self, wheel_dists, body_dists):
        """rover.py:663-668."""
        _lib.require_cuda(wheel_dists, body_dists)
        w = wheel_dists.to(torch.float16).contiguous()
        b = body_dists.to(torch.float16).contiguous()
        out = torch.empty(w.shape[0], dtype=torch.long, device=w.device)
        with torch.cuda.device(w.device):
            _lib.check(self._lib.rvb_check_collision(_lib.ptr(w), _lib.ptr(b), w.shape[0], _lib.ptr(out), self._stream()))
        self.rock_collison = out
        return out

    # ------------------------------------------------------------------ pre_physics_step, action part (rover.py:338-414)
    def pre_physics_step(self, actions) -> None:
        self.global_step += 1
        self.rover_loc, quat = self._rover.get_world_poses()
        self.rover_rot = tensor_quat_to_eul(quat)                   # used one step later by is_done (rover.py:343,615)
        reset_env_ids = self.reset_buf.nonzero(as_tuple=False).squeeze(-1)
        if len(reset_env_ids) > 0:
            self.reset_idx(reset_env_ids)
            self.set_targets(reset_env_ids)
        self.apply_actions(actions)

    def pre_physics_step_device(self, actions, max_attempts=64) -> None:
        """pre_physics_step (rover.py:338-414) with the reset path on the device: no reset_buf.nonzero(), no host-side goal
        loop -- one launch (rvb_reset_targets) resets the book-keeping of the envs whose reset_buf is set, draws their goals
        (Philox, keyed by (reset_seed, global_step, global env id)) until they clear the stones and looks their height up.
        Pose resets belong to the simulator: `self._rover.reset_idx_masked(reset_mask, initial_pos)` is called when the view
        provides it (the mask is a snapshot of reset_buf taken before it is cleared)."""
        self.global_step += 1
        self.rover_loc, quat = self._rover.get_world_poses()
        self.rover_rot = tensor_quat_to_eul(quat)
        self._reset_half(max_attempts=max_attempts)
        self.apply_actions(actions)

    def reset_targets_device(self, radius=8.0, thr=1.0, max_attempts=64, epoch=None, reset_mask=None):
        """reset_idx book-keeping + set_targets (rover.py:451-452, 566-584) for every env with reset_buf != 0, on the device.
        reset_mask: consume this mask instead (left untouched; reset_buf is then not cleared)."""
        hm = self.heightmap
        if self._shift_host is None:          # read once: a .cpu() per step would synchronise the stream
            self._shift_host = [float(v) for v in self.shift.flatten().cpu()]
        sh = self._shift_host
        with torch.cuda.device(torch.device(self._device)):
            _lib.check(self._lib.rvb_reset_targets(
                _lib.ptr(self.reset_buf if reset_mask is None else reset_mask), self.num_envs, int(self.env_offset), int(self.reset_seed),
                int(self.global_step if epoch is None else epoch), _lib.ptr(self.initial_pos), float(radius), _lib.ptr(self.stone_info),
                self.stone_info.shape[0], float(thr), int(max_attempts), _lib.ptr(hm), hm.shape[0], hm.shape[1],
                float(self.horizontal_scale), float(self.vertical_scale), float(sh[0]), float(sh[1]), _lib.ptr(self.target_positions),
                _lib.ptr(self.progress_buf), _lib.ptr(self.reset_buf if reset_mask is None else None), _lib.ptr(self.reset_counters),
                self.sem, self._stream()))
        return self.reset_counters

    def apply_actions(self, actions):
        """History push + Ackermann + joint-target mapping (rover.py:366-414)."""
        _actions = actions.to(self._device)
        if self.save_teacher_data:                                  # rover.py:373-375
            self._teacher_actions = _actions[:, 0:2].to(torch.float32)
        self.linear_velocity.input_state(_actions[:, 0])
        self.angular_velocity.input_state(_actions[:, 1])
        _, _, positions, velocities = Ackermann(_actions[:, 0], _actions[:, 1], self._device, sem=self.sem,
                                                want_targets=True)
        self.joint_position_targets, self.joint_velocity_targets = positions, velocities
        if hasattr(self._rover, "set_joint_position_targets"):
            self._rover.set_joint_position_targets(positions, indices=None,
                                                   joint_indices=getattr(self._rover, "actuated_pos_indices", None))
            self._rover.set_joint_velocity_targets(velocities, indices=None,
                                                   joint_indices=getattr(self._rover, "actuated_vel_indices", None))

    def reset_idx(self, env_ids):
        """Book-keeping half of rover.py:416-453 (pose resets belong to the simulator)."""
        if self.save_teacher_data:                                  # rover.py:420-422 (sets every env, as the reference does)
            self.reset_info[:] = 1
            self.reset_info[env_ids] = 1
        if hasattr(self._rover, "reset_idx"):
            self._rover.reset_idx(env_ids, self.initial_pos)
        self.reset_buf[env_ids] = 0
        self.progress_buf[env_ids] = 0

    # ------------------------------------------------------------------ calculate_metrics + is_done (rover.py:460-531,610-647)
    def _params(self):
        r = self.rew_scales
        return _lib.RewardParams(r["pos_reward"], r["heading_contraint_reward"], r["motion_contraint_reward"],
                                 r["goal_angle_reward"], r["boogie_contraint_reward"], self.max_episode_length,
                                 self.curriculum_level, self.num_envs_total, self.sem, 0)

    def _reward_reset(self):
        joints = self._rover.get_joint_positions().to(torch.float32).contiguous()
        lin, ang = self.linear_velocity.tracker, self.angular_velocity.tracker
        lin0, lin1 = lin[:, 0, 0].contiguous(), lin[:, 0, 1].contiguous()
        ang0, ang1 = ang[:, 0, 0].contiguous(), ang[:, 0, 1].contiguous()
        rot = self.rover_rot if self.rover_rot is not None else self.rover_rotation
        self._reset_next = torch.empty_like(self.reset_buf)
        p = self._params()
        e = self._ex
        with torch.cuda.device(torch.device(self._device)):
            _lib.check(self._lib.rvb_reward_reset(
                C.byref(p), _lib.ptr(self.rover_positions), _lib.ptr(self.target_positions), _lib.ptr(self.heading_diff),
                _lib.ptr(rot), _lib.ptr(lin0), _lib.ptr(lin1), _lib.ptr(ang0), _lib.ptr(ang1), _lib.ptr(joints),
                _lib.ptr(self.progress_buf), _lib.ptr(self.rock_collison if self.curriculum_level >= 2 else None),
                self.num_envs, _lib.ptr(self.rew_buf), _lib.ptr(self._reset_next), _lib.ptr(e["pos_reward"]),
                _lib.ptr(e["collision_penalty"]), _lib.ptr(e["uprightness_penalty"]),
                _lib.ptr(e["heading_contraint_penalty"]), _lib.ptr(e["motion_contraint_penalty"]),
                _lib.ptr(e["goal_angle_penalty"]), _lib.ptr(self.stats), _lib.ptr(self._stats_scratch), self._stream()))
        self._lin0, self._ang0 = lin0, ang0

    def calculate_metrics(self) -> None:
        """One fused launch computes the reward terms AND the next reset mask; is_done() publishes the mask."""
        self._reward_reset()
        self.extras.update(self._ex)
        self.extras["torque_penalty_driving"] = self._lin0          # rover.py:530-531
        self.extras["torque_penalty_steering"] = self._ang0

    def is_done(self) -> None:
        if self._reset_next is None:
            self._reward_reset()
        self.reset_buf[:] = self._reset_next
        self._reset_next = None

    # ------------------------------------------------------------------ goals / spawn validation (rover.py:533-584,649-661)
    def nearest_stone_edge(self, xy, thr):
        """-> (nearest f32 [M], flag i64 [M], count i32 [1] tensor); xy: [M,>=2] f32 with unit inner stride."""
        xy = xy if (xy.dim() == 2 and xy.stride(-1) == 1 and xy.dtype == torch.float32) else xy.float().contiguous()
        M = xy.shape[0]
        near = torch.empty(M, device=xy.device)
        flag = torch.empty(M, device=xy.device, dtype=torch.long)
        self._count.zero_()
        with torch.cuda.device(xy.device):
            _lib.check(self._lib.rvb_stone_validate(_lib.ptr(xy), xy.stride(0) if M > 1 else xy.shape[1], M,
                                                    _lib.ptr(self.stone_info), self.stone_info.shape[0], float(thr), 0,
                                                    _lib.ptr(near), _lib.ptr(flag), _lib.ptr(self._count), self._stream()))
        return near, flag, self._count

    def check_goal_collision(self, env_ids):
        _, flag, count = self.nearest_stone_edge(self.target_positions[env_ids][:, 0:2], 1.0)
        env_ids = flag * env_ids                                    # rover.py:540 (valid entries collapse to env 0)
        return env_ids, int(count.item())

    def generate_goals(self, env_ids, radius):
        reset_buf_len = 1
        while reset_buf_len > 0:
            self.random_goals(env_ids, radius=radius)
            env_ids, reset_buf_len = self.check_goal_collision(env_ids)

    def random_goals(self, env_ids, radius):
        num_sets = len(env_ids)
        alpha = 2 * math.pi * torch.rand(num_sets, device=self._device)
        self.target_positions[env_ids, 0] = radius * torch.cos(alpha) + 0 + self.initial_pos[env_ids, 0]
        self.target_positions[env_ids, 1] = radius * torch.sin(alpha) + 0 + self.initial_pos[env_ids, 1]

    def set_targets(self, env_ids):
        self.generate_goals(env_ids, radius=8)
        global_pos = self.target_positions[env_ids, 0:2]
        height = self.get_pos_height(self.heightmap, global_pos[:, 0:2], self.horizontal_scale, self.vertical_scale,
                                     self.shift[0:2])
        self.target_positions[env_ids, 2] = height

    def get_pos_height(self, heightmap, depth_points, horizontal_scale, vertical_scale, shift):
        _lib.require_cuda(heightmap, depth_points)
        hm = heightmap.to(torch.float32).contiguous()
        xy = depth_points
        xy = xy if (xy.dim() == 2 and xy.stride(-1) == 1 and xy.dtype == torch.float32) else xy.float().contiguous()
        M = xy.shape[0]
        sh = torch.as_tensor(shift).flatten().cpu()
        out = torch.empty(M, device=xy.device)
        with torch.cuda.device(xy.device):
            _lib.check(self._lib.rvb_height_lookup(_lib.ptr(hm), hm.shape[0], hm.shape[1], _lib.ptr(xy),
                                                   xy.stride(0) if M > 1 else xy.shape[1], M, float(horizontal_scale),
                                                   float(vertical_scale), float(sh[0]), float(sh[1]), _lib.ptr(out),
                                                   self.sem, self._stream()))
        return out

    def avoid_pos_rock_collision(self, curr_pos, max_iter=100000):
        """Whole fixed-point loop in one launch (no host sync per sweep).  Updates and returns curr_pos."""
        _lib.require_cuda(curr_pos)
        pos = curr_pos if (curr_pos.is_contiguous() and curr_pos.dtype == torch.float32) else curr_pos.float().contiguous()
        with torch.cuda.device(pos.device):
            _lib.check(self._lib.rvb_spawn_validate(_lib.ptr(pos), pos.shape[0], _lib.ptr(self.stone_info),
                                                    self.stone_info.shape[0], max_iter, _lib.ptr(self._count),
                                                    self._stream()))
        if pos is not curr_pos:
            curr_pos.copy_(pos)
        return curr_pos

    def set_initial_positions(self, positions):
        """set_up_scene's spawn validation (rover.py:214-219): stones, then terrain height + 0.5."""
        positions = self.avoid_pos_rock_collision(positions.clone().float().contiguous())
        h = self.get_pos_height(self.heightmap, positions[:, 0:2], self.horizontal_scale, self.vertical_scale,
                                self.shift[0:2])
        positions[:, 2] = h + 0.5
        self.initial_pos = positions
        return positions
