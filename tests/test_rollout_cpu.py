"""CPU tests of the rollout shim's host-side maths (normaliser with norm groups, policy head) against numpy restatements of
R/learning/normalizer.py and the actor construction of R/learning/pg_agent.py:140-160."""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
from deepmimic_b200.rollout import DeviceNormalizer, build_policy


def _np_normalizer_update(mean, mean_sq, count, x, groups, eps=0.02):
    new_mean, new_mean_sq = x.mean(0), (x * x).mean(0)

    def proc(new, old):
        out = new.copy()
        for g in np.unique(groups):
            idx = np.nonzero(groups == g)[0]
            if g == -1:
                out[idx] = old[idx]
            elif g != 0:
                out[idx] = new[idx].mean()
        return out
    new_mean, new_mean_sq = proc(new_mean, mean), proc(new_mean_sq, mean_sq)
    tot = count + x.shape[0]
    mean = count / tot * mean + x.shape[0] / tot * new_mean
    mean_sq = count / tot * mean_sq + x.shape[0] / tot * new_mean_sq
    std = np.maximum(np.sqrt(np.maximum(mean_sq - mean * mean, 0)), eps)
    return mean, mean_sq, tot, std


def test_normalizer_matches_reference_semantics():
    rng = np.random.default_rng(0)
    size = 12
    groups = np.array([-1, 0, 0, 0, 1, 1, 1, 2, 2, 0, 0, 0])
    n = DeviceNormalizer(size, groups)
    mean0, std0 = rng.normal(size=size), rng.uniform(0.5, 2, size=size)
    n.set_mean_std(mean0, std0)
    mean, mean_sq, count = mean0.copy(), std0 ** 2 + mean0 ** 2, 0
    for _ in range(3):
        x = rng.normal(1.0, 2.0, size=(50, size))
        n.record(torch.tensor(x, dtype=torch.float32))
        n.update()
        mean, mean_sq, count, std = _np_normalizer_update(mean, mean_sq, count, x, groups)
        np.testing.assert_allclose(n.mean.numpy(), mean, rtol=2e-5, atol=2e-5)
        np.testing.assert_allclose(n.std.numpy(), std, rtol=2e-4, atol=2e-5)
    assert n.mean[0].item() == pytest.approx(mean0[0])          # NORM_GROUP_NONE keeps its statistics (the phase slot)
    assert np.allclose(n.mean.numpy()[4:7], n.mean.numpy()[4])   # a shared group gets one mean
    x = torch.tensor(rng.normal(size=(5, size)), dtype=torch.float32)
    torch.testing.assert_close(n.unnormalize(n.normalize(x)), x, rtol=1e-5, atol=1e-5)


def test_policy_head_shapes_and_logp():
    torch.manual_seed(0)
    p = build_policy(227, 28, init_output_scale=0.01, noise=0.05)
    assert [l.weight.shape for l in p.hidden] == [(1024, 227), (512, 1024)] and p.mean.weight.shape == (28, 512)
    assert float(p.mean.weight.detach().abs().max()) <= 0.01 and float(p.logstd.detach()[0]) == pytest.approx(math.log(0.05))
    s = torch.randn(7, 227)
    mask = torch.tensor([1, 0, 1, 1, 0, 1, 1], dtype=torch.bool)
    a, logp = p.sample(s, mask)
    mu = p(s)
    torch.testing.assert_close(a[~mask], mu[~mask])               # non-exploring rows take the mode
    z = (a - mu) / p.logstd.exp()
    ref = (-0.5 * z * z - p.logstd - 0.5 * math.log(2 * math.pi)).sum(-1)
    torch.testing.assert_close(logp, ref, rtol=1e-4, atol=1e-4)


def _random_gated_actor(rng, s_dim=226, g_dim=3, a_dim=28, hidden=(1024, 512)):
    w = lambda i, o: (rng.standard_normal((i, o)) / math.sqrt(i)).astype(np.float32)
    b = lambda o: (0.1 * rng.standard_normal(o)).astype(np.float32)
    dims = [s_dim + g_dim] + list(hidden)
    return dict(hidden=[(w(i, o), b(o)) for i, o in zip(dims[:-1], dims[1:])], mean=(w(dims[-1], a_dim), b(a_dim)), logstd=b(a_dim),
                gate_common=(w(g_dim, 128), b(128)), gates=[dict(hidden=(w(128, 64), b(64)), bias=(w(64, h), b(h)), scale=(w(64, h), b(h))) for h in hidden],
                s_norm_mean=np.zeros(s_dim), s_norm_std=np.ones(s_dim), g_norm_mean=np.zeros(g_dim), g_norm_std=np.ones(g_dim),
                a_norm_mean=np.zeros(a_dim), a_norm_std=np.ones(a_dim))


def test_gated_policy_matches_numpy_restatement_of_the_reference_net():
    """build_gated_policy vs. a numpy restatement of fc_2layers_gated_1024units (R/learning/nets/fc_2layers_gated_1024units.py:6-58)."""
    import torch
    from deepmimic_b200.rollout import build_gated_policy, load_actor_weights
    from tests.test_task_scenes_cpu import _f64, gated_actor_mode
    rng = np.random.default_rng(4)
    actor = _random_gated_actor(rng)
    pol = load_actor_weights(build_gated_policy(226, 3, 28), actor).double()
    s, g = rng.standard_normal((5, 226)), rng.standard_normal((5, 3))
    with torch.no_grad():
        got = pol(torch.as_tensor(s), torch.as_tensor(g)).numpy()
    want = np.stack([gated_actor_mode(_f64(actor), s[i], g[i]) for i in range(5)])
    np.testing.assert_allclose(got, want, atol=1e-10)
    a, logp = pol.sample(torch.as_tensor(s), torch.as_tensor(g), explore_mask=torch.zeros(5, dtype=torch.bool))
    np.testing.assert_allclose(a.detach().numpy(), want, atol=1e-10)            # no exploration: the mode


def test_checkpoint_reader_returns_the_gate_layers_of_a_task_policy():
    import os
    from deepmimic_b200.assets import reference_root
    ref = reference_root()
    ckpt = os.path.join(ref or "", "data/policies/humanoid3d_amp/humanoid3d_amp_heading_locomotion.ckpt")
    if not ref or not os.path.exists(ckpt + ".index"):
        pytest.skip("reference checkout with pretrained policies not available (set DEEPMIMIC_REFERENCE_ROOT)")
    from deepmimic_b200.tf_checkpoint import load_actor
    a = load_actor(ckpt)
    assert [w.shape for w, _ in a["hidden"]] == [(229, 1024), (1024, 512)] and a["gate_common"][0].shape == (3, 128)
    assert [g["scale"][0].shape for g in a["gates"]] == [(64, 1024), (64, 512)] and a["g_norm_mean"].shape == (3,)


class _FakeEnv:
    """CPU stand-in with DeepMimicBatchEnv's surface, enough to exercise BatchedRollout.collect's control flow without a GPU."""

    def __init__(self, n, goal_size):
        import torch
        self.torch, self.num_envs, self.device, self.G = torch, n, torch.device("cpu"), goal_size
        self.t = torch.zeros(n)
        self.resets = 0
        self.done = torch.zeros(n, dtype=torch.bool)

    def get_state_size(self, agent_id=0): return 5
    def get_action_size(self, agent_id=0): return 2
    def get_goal_size(self, agent_id=0): return self.G
    def build_state_norm_groups(self, agent_id=0): return np.zeros(5, dtype=np.int32)
    def build_goal_norm_groups(self, agent_id=0): return np.zeros(self.G, dtype=np.int32)
    def build_state_offset(self, agent_id=0): return np.zeros(5)
    def build_state_scale(self, agent_id=0): return np.ones(5)
    def build_goal_offset(self, agent_id=0): return np.zeros(self.G)
    def build_goal_scale(self, agent_id=0): return np.ones(self.G)
    def build_action_offset(self, agent_id=0): return np.array([-1.0, 0.5])
    def build_action_scale(self, agent_id=0): return np.array([2.0, 4.0])

    def record_state(self, agent_id=0):
        return self.t[:, None] + self.torch.arange(5.0)[None, :]

    def record_goal(self, agent_id=0):
        return self.torch.stack([self.t, -self.t, self.torch.ones_like(self.t)], dim=1)[:, :self.G]

    def step(self, a):
        self.last_action = a.clone()
        self.t = self.t + 1.0
        self.done = self.t >= 3.0 + self.torch.arange(float(self.num_envs)) % 2      # episodes of 3 or 4 steps
        return self.record_state(), a.sum(dim=1), self.done.clone(), self.done.to(self.torch.int32)

    def reset(self, force_all=False):
        self.resets += int(self.done.sum())
        self.t = self.torch.where(self.done, self.torch.zeros_like(self.t), self.t)
        self.done = self.torch.zeros_like(self.done)


@pytest.mark.parametrize("goal_size", [0, 3])
def test_rollout_collect_control_flow_with_and_without_goals(goal_size):
    import torch
    from deepmimic_b200.rollout import BatchedRollout
    env = _FakeEnv(4, goal_size)
    ro = BatchedRollout(env, exp_rate=0.0, seed=1)
    assert type(ro.policy).__name__ == ("GatedGaussianMLPPolicy" if goal_size else "GaussianMLPPolicy")
    traj = ro.collect(9, record_stats=False)
    assert traj["states"].shape == (9, 4, 5) and traj["actions"].shape == (9, 4, 2) and traj["dones"].dtype == torch.bool
    assert ("goals" in traj) == (goal_size > 0)
    # episodes restart: env 0 (3 steps) is done at k = 2, 5, 8; env 1 (4 steps) at k = 3, 7
    assert traj["dones"][:, 0].nonzero().flatten().tolist() == [2, 5, 8] and traj["dones"][:, 1].nonzero().flatten().tolist() == [3, 7]
    assert env.resets == 3 + 2 + 3 + 2
    assert torch.equal(traj["states"][3, 0], torch.arange(5.0))                 # the state after a reset is re-recorded
    if goal_size:
        assert torch.equal(traj["goals"][4, 1], torch.tensor([0.0, -0.0, 1.0]))  # and so is the goal
    # exp_rate 0: the action is the un-normalised mode, a = mean_a + std_a * mu with mean = -offset, std = 1 / scale
    with torch.no_grad():
        s0 = traj["states"][0]
        mu = ro.policy(ro.s_norm.normalize(s0), ro.g_norm.normalize(traj["goals"][0])) if goal_size else ro.policy(ro.s_norm.normalize(s0))
    want = torch.tensor([1.0, -0.5]) + mu * torch.tensor([0.5, 0.25])
    assert torch.allclose(traj["actions"][0], want, atol=1e-6)
    assert torch.allclose(traj["rewards"][0], traj["actions"][0].sum(dim=1))
