"""Batched mirror of the reference's Python env surface (R/env/deepmimic_env.py:6-187, R/env/env.py:6-230) over the
C ABI.  Method names and meanings follow DeepMimicEnv; what was a per-agent vector there is an [N, .] CUDA tensor here
(N environments of this rank), and `agent_id` is accepted and ignored (the imitation scene has one agent).
For the unmodified single-env reference wrapper use the `DeepMimicCore` package next to this file instead."""
import numpy as np

from .capi import (BatchedCore, DM_ACTION_BOUND_MAX, DM_ACTION_BOUND_MIN, DM_ACTION_OFFSET, DM_ACTION_SCALE, DM_STATE_NORM_GROUPS,
                   DM_STATE_OFFSET, DM_STATE_SCALE)
from .sharding import StepExchange, pack_rows, rank_world, shard_range


class DeepMimicBatchEnv:
    class Terminate:
        Null, Fail, Succ = 0, 1, 2

    def __init__(self, args, num_envs, asset_root, device=0, seed=0, global_env_offset=0):
        import torch
        self.torch = torch
        self._core = BatchedCore(list(args), num_envs, asset_root, device=device, seed=seed, global_env_offset=global_env_offset)
        d = self._core.dims
        self.num_envs, self.device = d.num_envs, torch.device("cuda", device)
        self.stream = torch.cuda.ExternalStream(self._core.stream(), device=device)
        with torch.cuda.stream(self.stream):
            self._obs = torch.zeros(d.num_envs, d.state_size, device=self.device)
            self._rew = torch.zeros(d.num_envs, device=self.device)
            self._flags = torch.zeros(d.num_envs, 4, dtype=torch.int32, device=self.device)
        self._time = 0.0
        self._core.reset(True)

    # ---- stream ordering: the library works on its own stream; these two event waits make every method safe to call
    # from torch's current stream (inputs produced there are complete before the kernels read them, returned tensors are
    # complete before the caller's next op on that stream reads them).  No host synchronisation.
    def _pre(self):
        self.stream.wait_stream(self.torch.cuda.current_stream(self.device))

    def _post(self):
        self.torch.cuda.current_stream(self.device).wait_stream(self.stream)

    # ---- scene control (cDeepMimicCore::Update / Reset / GetTime, DeepMimicCore.cpp:88-139)
    def update(self, timestep, n_updates=1):
        self._core.update(timestep, n_updates)
        self._time += timestep * n_updates

    def reset(self, force_all=False):
        """Restarts finished episodes (every environment with force_all)."""
        self._pre()
        self._core.reset(force_all)

    def get_time(self):
        return self._time

    def get_name(self):
        """cScene::GetName of the configured scene (SceneImitate.cpp:209, SceneImitateAMP.cpp:211, SceneTargetAMP.cpp:233, ...)"""
        return self._core.scene_name()

    def is_rl_scene(self):
        return True

    def get_num_agents(self):
        return 1

    def get_num_update_substeps(self):
        return self._core.dims.num_update_substeps

    def set_mode(self, mode):
        self._core.set_mode(int(mode))

    def set_sample_count(self, count):
        """RLWorld feeds the learner's sample count back every iteration (R/learning/rl_agent.py -> env.set_sample_count):
        anneals the episode time limits of the following resets."""
        self._pre()
        self._core.set_sample_count(int(count))
        self._post()

    # ---- per-step queries; tensors are views of buffers rewritten by the next call
    def _refresh_flags(self):
        self._pre()
        self._core.flags(self._flags)
        self._post()
        return self._flags

    def need_new_action(self, agent_id=0):
        return self._refresh_flags()[:, 0].bool()

    def record_state(self, agent_id=0):
        self._pre()
        self._core.observe(self._obs, None)
        self._post()
        return self._obs

    def record_goal(self, agent_id=0):
        """[N, goal_size] float32 (goal_size 0 outside the AMP task scenes, 3 in target_amp / heading_amp)."""
        g = self._core.dims.goal_size
        if g == 0:
            return self.torch.zeros(self.num_envs, 0, device=self.device)
        if getattr(self, "_goal", None) is None:
            with self.torch.cuda.stream(self.stream):
                self._goal = self.torch.zeros(self.num_envs, g, device=self.device)
        self._pre()
        self._core.record_goal(self._goal)
        self._post()
        return self._goal

    def set_action(self, agent_id_or_actions, actions=None):
        a = agent_id_or_actions if actions is None else actions
        if tuple(a.shape) != (self.num_envs, self.get_action_size()) or a.dtype != self.torch.float32 or not a.is_cuda:
            raise ValueError("actions must be a float32 CUDA tensor [%d, %d]" % (self.num_envs, self.get_action_size()))
        self._pre()
        self._core.set_action(a.contiguous())

    def calc_reward(self, agent_id=0):
        self._pre()
        self._core.observe(None, self._rew)
        self._post()
        return self._rew

    # ---- AMP observations (R/env/deepmimic_env.py:147-166)
    def get_amp_obs_size(self):
        return self._core.dims.amp_obs_size

    def enable_amp_task_reward(self):
        return self._core.dims.goal_size > 0                # cSceneTargetAMP::EnableAMPTaskReward (SceneTargetAMP.cpp:222-225); false in imitate_amp

    def get_amp_obs_offset(self):
        return np.zeros(self.get_amp_obs_size())

    def get_amp_obs_scale(self):
        return np.ones(self.get_amp_obs_size())

    def get_amp_obs_norm_group(self):
        return np.zeros(self.get_amp_obs_size(), dtype=np.int32)

    def _amp_buf(self, which):
        # two buffers: the AMP agent fetches the agent's and the expert's observations of a step and stores both (R/learning/amp_agent.py:244-285)
        name = "_amp_" + which
        if not hasattr(self, name):
            with self.torch.cuda.stream(self.stream):
                setattr(self, name, self.torch.zeros(self.num_envs, self.get_amp_obs_size(), device=self.device))
        return getattr(self, name)

    def record_amp_obs_agent(self, agent_id=0):
        buf = self._amp_buf("agent")
        self._pre(); self._core.amp_obs_agent(buf); self._post()
        return buf

    def record_amp_obs_expert(self, agent_id=0, kin_time=None):
        buf = self._amp_buf("expert")
        self._pre(); self._core.amp_obs_expert(buf, kin_time); self._post()
        return buf

    def is_episode_end(self):
        return self._refresh_flags()[:, 1].bool()

    def check_terminate(self, agent_id=0):
        return self._refresh_flags()[:, 2]

    def check_valid_episode(self):
        return self._refresh_flags()[:, 3].bool()

    def step(self, actions, timestep=1.0 / 600.0):
        """One policy step: SetAction, the controller's query period worth of Update(timestep) calls (20 at the
        reference's 600 Hz / 30 Hz), then state, reward and flags.  Returns (obs, reward, done, terminate)."""
        self.set_action(actions)
        self.update(timestep, self._core.dims.updates_per_action)
        self._core.observe(self._obs, self._rew)
        f = self._refresh_flags()          # ends with _post(): obs / reward / flags are ordered before the caller's stream
        return self._obs, self._rew, f[:, 1].bool(), f[:, 2]

    # ---- sizes and normalisation statics (DeepMimicCore.cpp:246-330)
    def get_action_space(self, agent_id=0):
        return 0  # ActionSpace.Continuous

    def get_state_size(self, agent_id=0):
        return self._core.dims.state_size

    def get_goal_size(self, agent_id=0):
        return self._core.dims.goal_size

    def get_action_size(self, agent_id=0):
        return self._core.dims.action_size

    def get_num_actions(self, agent_id=0):
        return 0

    def build_state_offset(self, agent_id=0):
        return np.array(self._core.static(DM_STATE_OFFSET))

    def build_state_scale(self, agent_id=0):
        return np.array(self._core.static(DM_STATE_SCALE))

    def _task_kind(self):
        """0 none, 1 target_amp, 2 heading_amp, 3 heading_amp_getup, 4 strike_amp (dm_task.cuh: TaskKind)"""
        return int(self._core.task_params()[0][0]) if self._core.dims.goal_size > 0 else 0

    def build_goal_offset(self, agent_id=0):
        off = np.zeros(self._core.dims.goal_size)           # cRLSceneSimChar::BuildGoalOffsetScale (RLSceneSimChar.cpp:111-116)
        if self._task_kind() == 3:
            off[3] = -0.5                                   # the get-up phase (SceneHeadingAMPGetup.cpp:142-149)
        return off

    def build_goal_scale(self, agent_id=0):
        scl = np.ones(self._core.dims.goal_size)
        if self._task_kind() == 3:
            scl[3] = 2.0
        return scl

    def build_action_offset(self, agent_id=0):
        return np.array(self._core.static(DM_ACTION_OFFSET))

    def build_action_scale(self, agent_id=0):
        return np.array(self._core.static(DM_ACTION_SCALE))

    def build_action_bound_min(self, agent_id=0):
        return np.array(self._core.static(DM_ACTION_BOUND_MIN))

    def build_action_bound_max(self, agent_id=0):
        return np.array(self._core.static(DM_ACTION_BOUND_MAX))

    def build_state_norm_groups(self, agent_id=0):
        return np.array(self._core.static(DM_STATE_NORM_GROUPS), dtype=np.int32)

    def build_goal_norm_groups(self, agent_id=0):
        g = np.zeros(self._core.dims.goal_size, dtype=np.int32)      # gNormGroupSingle (RLSceneSimChar.cpp:136-140)
        kind = self._task_kind()
        if kind == 3:
            g[3] = -1                                                # gNormGroupNone for the get-up phase (SceneHeadingAMPGetup.cpp:151-157)
        elif kind == 4:
            g[:] = -1                                                # no normalisation of the strike goal (SceneStrikeAMP.cpp:401-405)
        return g

    def get_reward_min(self, agent_id=0):
        return 0.0

    def get_reward_max(self, agent_id=0):
        return 1.0

    def get_reward_fail(self, agent_id=0):
        return 0.0

    def get_reward_succ(self, agent_id=0):
        return 1.0

    def sync(self):
        self._core.sync()

    def counters(self):
        """(kernel launches so far, environments whose constraint solver ran out of row capacity).  The second number must stay 0: a
        truncated contact set is a silent deviation from the reference physics (DESIGN.md 5.5)."""
        return self._core.counters()

    def check_solver_capacity(self, raise_on_overflow=True):
        """Call at reset / collect boundaries (host synchronisation).  Raises (or warns) when any environment exceeded the solver's row
        capacity since the handle was created.  The capacity is fixed per character (DESIGN.md 5.5): treat the affected episodes as invalid."""
        over = self._core.counters()[1]
        if over:
            msg = "deepmimic_b200: %d environment(s) exceeded the contact-solver row capacity; contacts were truncated, so their episodes are invalid" % over
            if raise_on_overflow:
                raise RuntimeError(msg)
            import warnings
            warnings.warn(msg)
        return over


class ShardedDeepMimicEnv(DeepMimicBatchEnv):
    """One process per GPU: this rank owns shard_range(total_envs, rank, world) of the job's environments.  `step` keeps the base
    class's contract (the LOCAL rows: obs, reward, done, terminate -- what a replicated policy acts on); `step_gathered` additionally
    all-gathers every rank's [obs | reward | done] rows so that each rank (the learner) sees the whole job's transitions."""

    def __init__(self, args, total_envs, asset_root, seed=0):
        rank, world, local_rank = rank_world()
        off, cnt = shard_range(total_envs, rank, world)
        super().__init__(args, cnt, asset_root, device=local_rank, seed=seed, global_env_offset=off)
        self.rank, self.world, self.total_envs, self.env_offset = rank, world, total_envs, off
        S = self.get_state_size()
        with self.torch.cuda.stream(self.stream):
            self._rows = self.torch.zeros(cnt, S + 2, device=self.device)
            self._xchg = StepExchange(total_envs, S + 2, rank, world, self.device)

    def gather_rows(self, obs, rew, done):
        """local [cnt, .] rows -> the job's [total_envs, .] rows in global environment order (same on every rank)"""
        allrows = self._xchg.gather(pack_rows(self._rows, obs, rew, done))    # on the caller's stream, after _post()
        S = self.get_state_size()
        return allrows[:, :S], allrows[:, S], allrows[:, S + 1] > 0.5

    def step_gathered(self, actions, timestep=1.0 / 600.0):
        """step() for this rank's environments, then the all-gather: returns (local 4-tuple, (all_obs, all_reward, all_done))."""
        local = self.step(actions, timestep)
        return local, self.gather_rows(local[0], local[1], local[2])
