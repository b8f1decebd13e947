"""CPU tests of the oracle's restatement of the AMP task scenes (SURVEY 8f rank 2): cSceneTargetAMP / cSceneHeadingAMP goals, task
rewards, target updates and termination (R/DeepMimicCore/scenes/SceneTargetAMP.cpp, SceneHeadingAMP.cpp), the clip dataset of
cClipsController (anim/ClipsController.cpp) and the counter-based draw stream the CUDA path will share.  Known-answer tests against
independent numpy restatements of the cited formulas; behavioural pins with the reference's pretrained task policies.
The CUDA path does not run these scenes yet (dm_create refuses them): this is the oracle-first half of the row."""
import json
import math
import os

import numpy as np
import pytest

from deepmimic_b200.assets import reference_root
from tests.oracle_binding import Oracle

MINI = ["--motion_file", "data/datasets/test_clips_mini.txt"]
TARGET = MINI + ["--arg_file", "args/train_amp_target_humanoid3d_locomotion_args.txt"]
HEADING = MINI + ["--arg_file", "args/train_amp_heading_humanoid3d_locomotion_args.txt"]
MASK = (1 << 64) - 1


def u01(seed, a, b):
    """splitmix64 finaliser on seed + golden * (a * 2654435761 + b + 1) -> [0, 1): the stream of dm_policy.cu's u01."""
    z = (seed + 0x9E3779B97F4A7C15 * ((a * 2654435761 + b + 1) & MASK)) & MASK
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & MASK
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & MASK
    z ^= z >> 31
    return (z >> 11) * (1.0 / 9007199254740992.0)


class Stream:
    def __init__(self, seed, env, counter=0):
        self.seed, self.env, self.k = seed, env, counter

    def draw(self):
        v = u01(self.seed, self.env, self.k); self.k += 1
        return v

    def uniform(self, lo, hi):
        return lo if lo == hi else lo + self.draw() * (hi - lo)

    def coin(self, p):
        return self.uniform(0.0, 1.0) < p

    def normal(self, mean, std):
        u1, u2 = self.draw(), self.draw()
        return mean + std * math.sqrt(-2.0 * math.log(1.0 - u1)) * math.cos(2.0 * math.pi * u2)


def heading_of(pose):
    """cKinTree::CalcHeading (KinTree.cpp:1615-1627): rotate (1,0,0) by the root quaternion, heading = atan2(-z, x)."""
    w, x, y, z = pose[3:7]
    rx = 1 - 2 * (y * y + z * z); rz = 2 * (x * z - w * y)
    return math.atan2(-rz, rx)


def masses(asset_root):
    c = json.load(open(os.path.join(asset_root, "data/characters/humanoid3d.txt")))
    return np.array([b["Mass"] for b in c["BodyDefs"]])


def com_of(o, asset_root):
    m = masses(asset_root)
    return (m[:, None] * o.body_state()[0]).sum(0) / m.sum()


def step_policy(o, action=None, updates=20):
    o.set_action(np.zeros(o.action_size) if action is None else action)
    for _ in range(updates):
        o.update(1.0 / 600.0)


def test_stream_matches_the_documented_hash(asset_root):
    o = Oracle(TARGET, asset_root)
    for seed, a, b in [(0, 0, 0), (1, 2, 3), (0xDEADBEEF, 4095, 10 ** 6), (MASK, 7, 1 << 40)]:
        assert o.u01(seed, a, b) == u01(seed, a, b)
    xs = np.array([u01(5, 9, k) for k in range(20000)])
    assert 0.0 <= xs.min() and xs.max() < 1.0 and abs(xs.mean() - 0.5) < 0.01 and abs(xs.var() - 1 / 12.0) < 0.003


def test_clip_dataset_tables_and_sampler(asset_root):
    """cClipsController::LoadMotions / BuildClipsCDF / SelectNewMotion (ClipsController.cpp:145-236)."""
    o = Oracle(TARGET, asset_root)
    dur, w, cdf, loop = o.clip_table()
    assert o.num_clips() == 4 and list(w) == [20.0, 3.0, 1.0, 1.0]          # a missing "Weight" means 1
    np.testing.assert_allclose(cdf, np.cumsum(w) / w.sum(), rtol=1e-15)
    for f, d in zip(["run", "walk", "spinkick", "backflip"], dur):
        fr = json.load(open(os.path.join(asset_root, "data/motions/humanoid3d_%s.txt" % f)))["Frames"]
        assert d == pytest.approx(sum(x[0] for x in fr[:-1]), rel=1e-12)
    for u, want in [(0.0, 0), (0.79999, 0), (0.8, 1), (0.91, 1), (0.92, 2), (0.95999, 2), (0.96, 3), (0.999999, 3)]:
        assert o.select_clip(u) == want                                         # std::upper_bound: cdf[i] <= u moves on
    # a reset with an injected clip activates it: duration, cycle delta and the kinematic pose come from that clip
    for c in range(4):
        o.reset(0.2, 0.0, 20.0, clip=c)
        assert o.current_clip() == c and o.motion_duration == dur[c]
    o.reset(0.2, 0.0, 20.0)                                                     # no clip given: the active one stays
    assert o.current_clip() == 3
    # expert observations come from the sampled clip, not the active one (cSceneImitateAMP::SampleExpertMotion, SceneImitateAMP.cpp:260-277)
    e0, e1 = o.record_amp_obs_expert(0.3, clip=0), o.record_amp_obs_expert(0.3, clip=1)
    assert np.isfinite(e0).all() and np.abs(e0 - e1).max() > 1e-2
    single = Oracle(["--arg_file", "args/train_humanoid3d_walk_args.txt", "--scene", "imitate_amp", "--enable_amp_obs_local_root", "true"], asset_root)
    es = single.record_amp_obs_expert(0.3)                                      # clip 1 is the walk clip
    keep = np.ones(226, dtype=bool); keep[[0, 71]] = False                       # root heights are relative to each kinematic character's own origin height
    np.testing.assert_allclose(es[keep], e1[keep], atol=1e-12)


@pytest.mark.parametrize("args,size", [(TARGET, 3), (HEADING, 3), (["--arg_file", "args/train_humanoid3d_walk_args.txt"], 0)])
def test_goal_size_and_task_reward_flag(asset_root, args, size):
    o = Oracle(args, asset_root)
    assert o.goal_size == size and o.enable_amp_task_reward() == (size > 0)
    assert o.state_size == (226 if size else 227) and o.amp_obs_size() == 226


def test_reset_draw_order_target(asset_root):
    """cSceneTargetAMP::Reset (SceneTargetAMP.cpp:129-134): timer max ~ U(5, 10), then target = root + dist (cos, 0, sin) with
    dist ~ U(0, max_target_dist), theta ~ U(0, 2 pi) (SceneTargetAMP.cpp:259-274)."""
    o = Oracle(TARGET, asset_root)
    o.set_task_stream(77, 12, 0)
    o.reset(0.25, 1.1, 20.0, clip=1)
    s = Stream(77, 12)
    tmax = s.uniform(5.0, 10.0); dist = s.uniform(0.0, 10.0); th = s.uniform(0.0, 2 * math.pi)
    t = o.task_state()
    root = o.get_pose()[0][:3]
    assert t["timer"] == 0.0 and t["timer_max"] == pytest.approx(tmax, rel=1e-15) and o.task_counter() == 3
    np.testing.assert_allclose(t["target_pos"], [root[0] + dist * math.cos(th), 0.0, root[2] + dist * math.sin(th)], atol=1e-12)
    assert t["target_speed"] == 1.0 and np.all(t["prev_action_com"] == 0.0)      # DeepMimicCharController.cpp:227-228


def test_target_goal_and_reward_known_answers(asset_root):
    o = Oracle(TARGET, asset_root)
    o.set_task_stream(3, 0, 0)
    o.reset(0.4, -2.0, 20.0, clip=0)
    step_policy(o); step_policy(o)                                                # prev-action bookkeeping is live now
    pose = o.get_pose()[0]
    root, hd = pose[:3], heading_of(pose)
    com = com_of(o, asset_root)
    np.testing.assert_allclose(o.calc_com(), com, atol=1e-12)
    t = o.task_state()
    # cDeepMimicCharController::UpdateCalcTau advances the clock BEFORE HandleNewAction stamps it (DeepMimicCharController.cpp:71-78,262-267), so
    # at the next query the step lasted 19 updates on that clock while the COM moved for 20: the reference's average speed runs 20/19 high
    dt_step = 19 / 600.0
    vel_terms = []
    vel = (com - t["prev_action_com"]) / dt_step; vel[1] = 0.0                    # planar COM velocity on the controller's clock
    ang = math.atan2(vel[2], vel[0]) + math.acos(0.5 / np.linalg.norm(vel))       # a direction along which the COM moves at 0.5 m/s
    partial = [com[0] + 4.0 * math.cos(ang), 0.0, com[2] + 4.0 * math.sin(ang)]
    for tar in ([root[0] + 3.0, 0.0, root[2] - 1.5], [root[0] - 0.2, 0.0, root[2] + 0.1], [root[0] + 14.0, 0.0, root[2] + 6.0], [root[0], 0.0, root[2]], partial):
        tar = np.array(tar)
        o.set_task_state(tar, 1.0, 0.0, t["timer"], t["timer_max"], t["prev_action_com"])
        rel = tar - root; rel[1] = 0.0
        dist = np.linalg.norm(rel)
        # RecordGoal (SceneTargetAMP.cpp:185-215): direction in the heading frame, then the distance
        if dist > 1e-4:
            c, s_ = math.cos(-hd), math.sin(-hd)                                 # rotation about +y by -heading
            loc = np.array([c * rel[0] + s_ * rel[2], 0.0, -s_ * rel[0] + c * rel[2]]) / dist
        else:
            loc = np.array([1.0, 0.0, 0.0])
        np.testing.assert_allclose(o.record_goal(), [loc[0], loc[2], dist], atol=1e-12)
        # CalcReward (SceneTargetAMP.cpp:3-80)
        fail = dist * dist > 15.0 ** 2
        if fail:
            want = 0.0
        else:
            pos_r = math.exp(-0.5 * dist * dist)                                 # --pos_reward_scale 0.5
            if dist * dist < 0.25:
                vel_r = 1.0
            else:
                d = tar - com; d[1] = 0.0
                dirn = d / np.linalg.norm(d)
                avg_vel = float(dirn @ (com - t["prev_action_com"])) / dt_step
                err = max(1.0 - avg_vel, 0.0)                                    # --enable_min_tar_vel true, --tar_speed 1
                vel_r = 0.0 if avg_vel < 0 else math.exp(-4.0 * err * err)
                vel_terms.append(vel_r)
            want = 0.6 * pos_r + 0.4 * vel_r
        assert o.calc_reward() == pytest.approx(want, abs=1e-9)
        assert o.check_terminate() == (1 if fail else 0) and o.check_target_succ() == (dist < 0.5)   # SceneTargetAMP.cpp:171-183,281-319
    assert any(0.0 < v < 1.0 for v in vel_terms), vel_terms                        # the velocity branch was exercised non-trivially
    # moving away from the target: no velocity reward
    away = com + 5.0 * (t["prev_action_com"] - com) / np.linalg.norm((t["prev_action_com"] - com)[[0, 2]])
    o.set_task_state([away[0], 0.0, away[2]], 1.0, 0.0, t["timer"], t["timer_max"], t["prev_action_com"])
    d2 = (away[0] - root[0]) ** 2 + (away[2] - root[2]) ** 2
    assert o.calc_reward() == pytest.approx(0.6 * math.exp(-0.5 * d2), abs=1e-9)


def test_heading_goal_reward_and_update_sequence(asset_root):
    o = Oracle(HEADING, asset_root)
    o.set_task_stream(11, 5, 0)
    o.reset(0.1, 0.7, 20.0, clip=0)
    s = Stream(11, 5)
    tmax = s.uniform(0.2, 0.5)
    s.uniform(0.0, 10.0); s.uniform(0.0, 2 * math.pi)                             # the (unused) target position is still drawn: mEnableRandTargetPos stays true
    speed = s.uniform(1.0, 5.0)
    t = o.task_state()
    assert t["timer_max"] == pytest.approx(tmax, rel=1e-15) and t["target_speed"] == pytest.approx(speed, rel=1e-15) and t["target_heading"] == 0.0
    # replay 3 s of target updates (SceneTargetAMP.cpp:136-145,232-246; SceneHeadingAMP.cpp:148-205) against the stream
    heading, timer = 0.0, 0.0
    changes = 0
    for k in range(1800):
        o.update(1.0 / 600.0)
        timer += 1.0 / 600.0
        if timer >= tmax:
            s.uniform(0.0, 10.0); s.uniform(0.0, 2 * math.pi)                     # ResetTargetPos
            heading += s.uniform(-math.pi, math.pi) if s.coin(0.01) else s.normal(0.0, 0.15)
            if s.coin(0.02):
                speed = min(max(s.uniform(1.0, 5.0), 1.0), 5.0)
            timer, tmax = 0.0, s.uniform(0.2, 0.5)
            changes += 1
        t = o.task_state()
        assert t["target_heading"] == pytest.approx(heading, abs=1e-12) and t["target_speed"] == pytest.approx(speed, rel=1e-15)
        assert t["timer"] == pytest.approx(timer, abs=1e-12) and t["timer_max"] == pytest.approx(tmax, rel=1e-15)
    assert changes >= 5 and o.task_counter() == s.k
    # goal (SceneHeadingAMP.cpp:136-151) and reward (SceneHeadingAMP.cpp:3-48) at a need-new-action boundary
    o.reset(0.1, 0.7, 20.0, clip=1)
    step_policy(o); step_policy(o)
    pose = o.get_pose()[0]
    t = o.task_state()
    com = com_of(o, asset_root)
    for th, spd in [(0.0, 1.0), (1.3, 2.5), (-2.0, 4.0), (math.pi, 1.5)]:
        o.set_task_state(t["target_pos"], spd, th, t["timer"], t["timer_max"], t["prev_action_com"])
        rel = th - heading_of(pose)
        np.testing.assert_allclose(o.record_goal(), [math.cos(rel), -math.sin(rel), spd], atol=1e-12)
        v = (com - t["prev_action_com"]) / (19 / 600.0); v[1] = 0.0                  # 19, not 20: see the target test
        sp = math.cos(th) * v[0] - math.sin(th) * v[2]
        want = math.exp(-0.25 * (spd - sp) ** 2) if sp > 0 else 0.0              # --vel_reward_scale 0.25, enable_min_tar_vel false here
        assert o.calc_reward() == pytest.approx(want, abs=1e-9)
    assert o.check_terminate() == 0                                               # no distance failure in the heading scene


def test_task_scenes_keep_the_action_history_across_resets(asset_root):
    """cSceneTargetAMP::Reset calls cSceneImitate::Reset, not cSceneImitateAMP::Reset (SceneTargetAMP.cpp:129-134): no InitHist, the
    previous-pose half of the agent observation stays the state at the last applied action.  imitate_amp re-initialises it from the clip."""
    pose_size = 71                                                                # 71 pose + 42 vel floats per time step (SceneImitateAMP.cpp:214-258)
    for args, keeps in ((TARGET, True), (["--scene", "imitate_amp", "--arg_file", "args/train_humanoid3d_walk_args.txt"], False)):
        o = Oracle(args, asset_root)
        o.set_task_stream(1, 0, 0)
        o.reset(0.3, 0.0, 20.0)
        step_policy(o); step_policy(o, updates=7)
        before = o.record_amp_obs_agent()[pose_size:2 * pose_size]
        o.reset(0.9, 0.0, 20.0)
        after = o.record_amp_obs_agent()[pose_size:2 * pose_size]
        same = np.allclose(before[7:-12], after[7:-12], atol=1e-12)               # joint rotations of the history pose (heading-frame free)
        assert same == keeps


def _f64(a):
    if isinstance(a, dict):
        return {k: _f64(v) for k, v in a.items()}
    if isinstance(a, (list, tuple)):
        return type(a)(_f64(v) for v in a)
    return np.asarray(a, dtype=np.float64)


def gated_actor_mode(actor, s, g):
    """fc_2layers_gated_1024units (R/learning/nets/fc_2layers_gated_1024units.py:6-58) + Gaussian mode, numpy."""
    relu = lambda x: np.maximum(x, 0.0)
    ns = (s - actor["s_norm_mean"]) / actor["s_norm_std"]; ng = (g - actor["g_norm_mean"]) / actor["g_norm_std"]
    gc = relu(ng @ actor["gate_common"][0] + actor["gate_common"][1])
    h = np.concatenate([ns, ng], axis=-1)
    for (w, b), gt in zip(actor["hidden"], actor["gates"]):
        gh = relu(gc @ gt["hidden"][0] + gt["hidden"][1])
        scale = 2.0 / (1.0 + np.exp(-(gh @ gt["scale"][0] + gt["scale"][1])))
        h = relu(scale * (h @ w + b) + gh @ gt["bias"][0] + gt["bias"][1])
    return (h @ actor["mean"][0] + actor["mean"][1]) * actor["a_norm_std"] + actor["a_norm_mean"]


# the committed archive's 56-entry clip dataset (the reference's locomotion dataset has 56 clips but is not in the archive): the reset
# clip ids of the policy pins below exist in it, and its clips are the archive's walk / run clips
SYNTH56 = ["--motion_file", "data/datasets/synthetic_locomotion_56.txt"]


def run_task_policy(asset_root, task, arg_file, seed, clip, t0, theta, steps=600):
    a = fixture_task_actor(task)
    o = Oracle(SYNTH56 + ["--arg_file", arg_file], asset_root)
    o.L.dmo_set_mode(o.h, 1)
    o.set_task_stream(seed, 0, 0)
    o.reset(t0, theta, 20.0, clip=clip)
    rew, succ, dist = [], 0, []
    for _ in range(steps):
        if o.is_episode_end():
            break
        g = o.record_goal()
        dist.append(g[2])
        o.set_action(gated_actor_mode(a, o.record_state(), g))
        for _ in range(20):
            o.update(1.0 / 600.0)
            if o.is_episode_end():
                break
        rew.append(o.calc_reward())
        succ += o.check_target_succ()
    return len(rew), float(np.mean(rew)), o.has_fallen(), succ, np.array(dist), o


needs_reference = pytest.mark.skipif(not (reference_root() and os.path.exists(os.path.join(reference_root(), "data/policies/humanoid3d_amp/humanoid3d_amp_strike_walk_punch.ckpt.index"))),
                                     reason="reference checkout with pretrained policies not available (set DEEPMIMIC_REFERENCE_ROOT)")


@pytest.mark.parametrize("seed,clip,t0,theta", [(1, 0, 0.3, 0.4), (2, 30, 1.0, -2.5)])
def test_pretrained_target_policy_walks_to_its_targets_in_the_oracle(asset_root, seed, clip, t0, theta):
    """The reference's own target-location policy (fp16 fixture; trained in the real simulator on goals from the real RecordGoal) reaches the
    targets the oracle draws: it spends a good part of the 20 s inside the 0.5 m success radius and never falls.  A wrong goal frame, sign or
    target update would send it elsewhere."""
    n, mean_r, fallen, succ, dist, o = run_task_policy(asset_root, "target", "args/train_amp_target_humanoid3d_locomotion_args.txt", seed, clip, t0, theta)
    assert n == 600 and not fallen, (n, fallen)
    assert succ >= 60 and dist.min() < 0.2 and mean_r > 0.4, (succ, dist.min(), mean_r)


@pytest.mark.parametrize("seed,clip,t0,theta", [(1, 0, 0.3, 0.4), (5, 17, 0.5, 2.0)])
def test_pretrained_heading_policy_follows_heading_and_speed_in_the_oracle(asset_root, seed, clip, t0, theta):
    """Same for the heading policy: the task reward exp(-0.25 (v* - v)^2) of the oracle's heading / speed commands stays high for 20 s."""
    n, mean_r, fallen, succ, dist, o = run_task_policy(asset_root, "heading", "args/train_amp_heading_humanoid3d_locomotion_args.txt", seed, clip, t0, theta)
    assert n == 600 and not fallen, (n, fallen)
    assert mean_r > 0.8, mean_r


# ------------------------------------------------------------------------------------------------ device-side task logic, run on the host
@pytest.fixture(scope="module")
def task_shim(tmp_path_factory):
    """deepmimic_b200/csrc/kernels/dm_task.cuh (what the TASK instantiation of dm_step_kernel and the dm_task_* kernels execute per
    environment) compiled with g++ through tests/task_shim.cpp."""
    import ctypes as C
    import subprocess
    here = os.path.dirname(os.path.abspath(__file__))
    so = str(tmp_path_factory.mktemp("shim") / "libtask_shim.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", os.path.join(here, "task_shim.cpp"), "-o", so])
    L = C.CDLL(so)
    d, dp_, u64 = C.c_double, C.POINTER(C.c_double), C.c_uint64
    L.shim_reset.argtypes = [dp_, dp_, u64, u64, d, d]
    L.shim_update.argtypes = [dp_, dp_, u64, u64, d, d, d]
    L.shim_dist_fail.argtypes = [dp_, dp_, d, d]
    L.shim_goal.argtypes = [dp_, dp_, d, d, d, dp_]
    L.shim_reward.argtypes = [dp_, dp_, C.c_int, d, d, d]
    L.shim_reward.restype = d
    return L


def _ptr(a):
    import ctypes as C
    return a.ctypes.data_as(C.POINTER(C.c_double))


@pytest.mark.parametrize("args", [TARGET, HEADING])
def test_device_task_logic_matches_the_oracle_on_the_host(asset_root, task_shim, args, monkeypatch):
    """Drives dm_task.cuh (host build) with the oracle's root positions and compares the whole task block, the goal, the reward and the
    distance failure with the oracle after every update of a 6 s episode under a random policy.  Also checks that the C-ABI host loader
    fills the scene constants the device code receives."""
    from deepmimic_b200 import capi
    monkeypatch.setenv("DM_EXPERIMENTAL_TASK_SCENES", "1")
    single = ["--kin_ctrl", "motion", "--motion_file", "data/motions/humanoid3d_run.txt"] + args[2:]   # the device path takes one clip for now
    if args is TARGET:
        single = ["--rand_target_time_min", "1", "--rand_target_time_max", "2", "--tar_fail_dist", "6"] + single   # several re-targets and a distance failure in 6 s
    hm = capi.HostModel(single, asset_root)
    P, _, _ = hm.task_params()
    assert hm.dims.goal_size == 3 and P[0] == (1 if args is TARGET else 2)
    o = Oracle(single, asset_root)
    seed, env = 99, 1234
    o.set_task_stream(seed, env, 0)
    o.reset(0.2, 0.9, 20.0)
    t = np.zeros(16)
    root = o.get_pose()[0][:3]
    task_shim.shim_reset(_ptr(P), _ptr(t), seed, env, root[0], root[2])

    def compare():
        ts = o.task_state()
        want = np.array([ts["target_pos"][0], ts["target_pos"][2], ts["target_speed"], ts["target_heading"], ts["timer"], ts["timer_max"]])
        # the reset target hangs off cSimCharacter::GetRootPos (float Bullet state); the shim is fed the double pose the oracle was reset with
        np.testing.assert_allclose(t[:2], want[:2], rtol=0, atol=1e-7)
        np.testing.assert_allclose(t[2:6], want[2:], rtol=0, atol=1e-12)
        assert int(t[12]) == o.task_counter()
    compare()
    rng = np.random.default_rng(0)
    st = o.action_statics()
    n_goal = n_far = 0
    for k in range(3600):
        if o.need_new_action():
            pose = o.get_pose()[0]
            com = o.calc_com()
            ts = o.task_state()
            t[6:9] = ts["prev_action_com"]; t[9:12] = com
            g = np.zeros(3)
            task_shim.shim_goal(_ptr(P), _ptr(t), pose[0], pose[2], heading_of(pose), _ptr(g))
            np.testing.assert_allclose(g, o.record_goal(), atol=1e-12)
            if k > 0:
                r = task_shim.shim_reward(_ptr(P), _ptr(t), int(o.has_fallen()), pose[0], pose[2], 19.0 / 600.0)
                assert r == pytest.approx(o.calc_reward(), abs=1e-9)
            n_goal += 1
            o.set_action(np.clip(-st[0] + 0.1 / st[1] * rng.standard_normal(o.action_size), st[2], st[3]))
        o.update(1.0 / 600.0)
        root = o.get_pose()[0][:3]
        task_shim.shim_update(_ptr(P), _ptr(t), seed, env, 1.0 / 600.0, root[0], root[2])
        compare()
        tp = o.task_state()["target_pos"]
        too_far = args is TARGET and (root[0] - tp[0]) ** 2 + (root[2] - tp[2]) ** 2 > P[5] ** 2
        assert task_shim.shim_dist_fail(_ptr(P), _ptr(t), root[0], root[2]) == (1 if too_far else 0)
        if too_far:
            n_far += 1
            assert o.check_terminate() == 1
    assert n_goal == 180 and o.task_counter() > (3 if args is TARGET else 50) and (n_far > 0) == (args is TARGET)


def test_unvalidated_task_scenes_stay_refused_without_the_opt_in(asset_root, monkeypatch):
    """target_amp / heading_amp are on the default path since round 2 (validated on hardware); heading_amp_getup / strike_amp and every other
    scene name are still refused unless DM_EXPERIMENTAL_TASK_SCENES=1."""
    from deepmimic_b200 import capi
    monkeypatch.delenv("DM_EXPERIMENTAL_TASK_SCENES", raising=False)
    for bad in (GETUP, STRIKE, ["--scene", "dribble_amp"] + TARGET, ["--scene", "kin_char"] + TARGET):
        with pytest.raises(RuntimeError, match="Unsupported scene"):
            capi.HostModel(bad, asset_root)
    assert capi.HostModel(HEADING, asset_root).dims.goal_size == 3
    m = capi.HostModel(TARGET, asset_root)                                      # the mini dataset (4 clips) loads in a task scene ...
    monkeypatch.setenv("DM_EXPERIMENTAL_TASK_SCENES", "1")
    assert m.dims.goal_size == 3
    dur, cdf = m.clip_table()
    o = Oracle(TARGET, asset_root)
    np.testing.assert_array_equal(dur, o.clip_table()[0]); np.testing.assert_array_equal(cdf, o.clip_table()[2])
    # the get-up and strike scenes load too (goal size 4) and the loader hands the device the constants the host-checked logic was tested with
    g = capi.HostModel(GETUP, asset_root)
    Pg, _, _ = g.task_params()
    assert g.dims.goal_size == 4 and Pg[0] == 3
    np.testing.assert_allclose(Pg[16:48], _ext_params(getup_time=max(dur[1], dur[2]), root_h=1.2, head_h=2.0, head_id=2), atol=0)
    k = capi.HostModel(STRIKE, asset_root)
    Pk, _, _ = k.task_params()
    assert k.dims.goal_size == 4 and Pk[0] == 4
    np.testing.assert_allclose(Pk[16:48], _ext_params(head_id=0, strike=(8,), fail=(0, 1, 2), init_hit=0.1), atol=0)
    np.testing.assert_allclose(Pk[:7], [4, 5.0, 10.0, 10.0, 0.5, 15.0, 0.5], atol=0)   # kind, target timer, max / success / fail distance, pos reward scale
    np.testing.assert_allclose(Pk[13:15], [1.0, 1.0], atol=0)                          # tar_speed, enable_min_tar_vel
    with pytest.raises(RuntimeError, match="strike_amp needs --strike_bodies"):
        capi.HostModel(["--scene", "strike_amp"] + TARGET, asset_root)
    with pytest.raises(RuntimeError, match="more than one clip"):               # ... but not in the plain AMP imitation scene
        capi.HostModel(["--scene", "imitate_amp"] + TARGET, asset_root)


@pytest.mark.parametrize("sync_rot", [True, False])
def test_device_clip_wrap_sync_matches_the_oracle_on_the_host(asset_root, task_shim, sync_rot):
    """kin_wrap_sync (dm_task.cuh; what dm_step_kernel<.., kVarRootRot> runs at a clip wrap) against the oracle's SyncKinCharNewCycle: the
    character is turned by 0.7 rad and drifts until the walk clip wraps; the routine gets the pre-update clocks, origin and simulated base
    state from the oracle's snapshot and the fp32 clip table the device holds, and must reproduce the oracle's origin after that update."""
    import ctypes as C
    args = ["--sync_char_root_rot", "true" if sync_rot else "false", "--arg_file", "args/train_humanoid3d_walk_args.txt"]
    o = Oracle(args, asset_root)
    o.reset(0.2, 0.0, 20.0)
    p, v = o.get_pose()
    c, s_ = math.cos(0.35), math.sin(0.35)
    w, x, y, z = p[3:7]
    p[3:7] = [c * w - s_ * y, c * x + s_ * z, c * y + s_ * w, c * z - s_ * x]
    o.set_pose_vel(p, v)
    # the clip table as the device stores it: fp32 frames, root x / z recentred on frame 0, quaternions normalised, cumulative frame times
    fr = np.array(json.load(open(os.path.join(asset_root, "data/motions/humanoid3d_walk.txt")))["Frames"], dtype=np.float64)
    times = np.concatenate([[0.0], np.cumsum(fr[:-1, 0])])
    frames = fr[:, 1:].copy()
    frames[:, 0] -= frames[0, 0]; frames[:, 2] -= frames[0, 2]
    frames[:, 3:7] /= np.linalg.norm(frames[:, 3:7], axis=1, keepdims=True)
    f32 = np.ascontiguousarray(frames, dtype=np.float32)
    cyc_delta = np.array([f32[-1, 0] - f32[0, 0], 0.0, f32[-1, 2] - f32[0, 2]], dtype=np.float32)
    dur = o.motion_duration
    assert dur == pytest.approx(times[-1], rel=1e-12)
    task_shim.shim_wrap_sync.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_float), C.c_int, C.c_int, C.POINTER(C.c_float), C.c_double, C.c_double,
                                         C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_double, C.c_double, C.POINTER(C.c_double), C.c_int, C.c_int]
    nj, scale = o.num_joints, 4.0
    clk = 13 + 55 * nj
    wraps = 0
    for k in range(int(2.2 * dur * 600)):
        pre = o.get_snapshot()
        kin_time = pre[clk] + 1.0 / 600.0
        wrap = (kin_time / dur) % 1.0 < (pre[clk] / dur) % 1.0
        o.update(1.0 / 600.0)
        if not wrap:
            continue
        wraps += 1
        origin = pre[clk + 1: clk + 4].copy(); origin_rot = pre[clk + 4: clk + 8].copy()
        simq = pre[3:7].copy()
        task_shim.shim_wrap_sync(_ptr(times), f32.ctypes.data_as(C.POINTER(C.c_float)), f32.shape[1], f32.shape[0], cyc_delta.ctypes.data_as(C.POINTER(C.c_float)),
                                 dur, kin_time, _ptr(origin), _ptr(origin_rot), pre[0] / scale, pre[2] / scale, _ptr(simq), 1, 1 if sync_rot else 0)
        post = o.get_snapshot()
        np.testing.assert_allclose(origin, post[clk + 1: clk + 4], atol=1e-5)       # the oracle reads the root through float link frames
        np.testing.assert_allclose(origin_rot, post[clk + 4: clk + 8], atol=1e-5)
        turned = abs(2 * math.atan2(post[clk + 6], post[clk + 4]))
        assert (turned > 0.3) == sync_rot
    assert wraps == 2


def fixture_task_actor(task):
    """tests/golden/policy_humanoid3d_amp_<task>_locomotion_fp16.npz (tests/golden/make_policy_fixture.py) in load_actor's layout."""
    name = dict(target="target_locomotion", heading="heading_locomotion", heading_getup="heading_getup_locomotion_getup", strike="strike_walk_punch")[task]
    f = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "policy_humanoid3d_amp_%s_fp16.npz" % name))
    g = lambda k: f[k].astype(np.float64)
    return dict(hidden=[(g("w0"), g("b0")), (g("w1"), g("b1"))], mean=(g("wm"), g("bm")), logstd=g("logstd"), gate_common=(g("gcw"), g("gcb")),
                gates=[dict(hidden=(g("g%d_hidden_w" % i), g("g%d_hidden_b" % i)), bias=(g("g%d_bias_w" % i), g("g%d_bias_b" % i)),
                            scale=(g("g%d_scale_w" % i), g("g%d_scale_b" % i))) for i in range(2)],
                s_norm_mean=g("s_mean"), s_norm_std=g("s_std"), g_norm_mean=g("g_mean"), g_norm_std=g("g_std"), a_norm_mean=g("a_mean"), a_norm_std=g("a_std"))


@pytest.mark.parametrize("task,args,clip", [("target", TARGET, 0), ("heading", HEADING, 1)])
def test_fixture_task_policies_in_the_oracle_without_the_reference_tree(asset_root, task, args, clip):
    """Hermetic version of the pretrained-policy pins: fp16 fixtures of the two task policies, the committed asset archive and its mini clip
    dataset.  Target: the policy walks into the 0.5 m success radius of the oracle's targets; heading: the velocity reward stays high."""
    a = fixture_task_actor(task)
    o = Oracle(args, asset_root)
    o.L.dmo_set_mode(o.h, 1)
    o.set_task_stream(4, 0, 0)
    o.reset(0.3, 0.4, 20.0, clip=clip)
    rew, succ = [], 0
    for _ in range(600):
        if o.is_episode_end():
            break
        o.set_action(gated_actor_mode(a, o.record_state(), o.record_goal()))
        for _ in range(20):
            o.update(1.0 / 600.0)
            if o.is_episode_end():
                break
        rew.append(o.calc_reward())
        succ += o.check_target_succ()
    assert len(rew) == 600 and not o.has_fallen()
    if task == "target":
        assert succ >= 60 and np.mean(rew) > 0.4, (succ, np.mean(rew))      # measured: 161 steps inside the radius, mean 0.60
    else:
        assert np.mean(rew) > 0.85, np.mean(rew)                              # measured: 0.96


# ------------------------------------------------------------------------------------------------ heading_amp_getup (cSceneHeadingAMPGetup)
# the logic does not care what the flagged clips show: clips 1 and 2 of the mini dataset stand in for the get-up motions
GETUP = ["--scene", "heading_amp_getup", "--getup_motion_ids", "1", "2", "--getup_height_root", "1.2", "--getup_height_head", "2.0", "--head_id", "2"] + HEADING   # heights above a standing character: unsaturated reward


def test_getup_goal_reward_and_timer_known_answers(asset_root):
    """SceneHeadingAMPGetup.cpp: goal = heading goal + get-up phase (:125-140,289-294), get-up reward (:18-38), timer sync with a get-up clip at
    reset (:179-199), no contact fall while getting up (:256-265)."""
    o = Oracle(GETUP, asset_root)
    dur = o.clip_table()[0]
    T = max(dur[1], dur[2])
    assert o.goal_size == 4 and o.getup_state()["getup_time"] == T
    o.set_task_stream(2, 0, 0)
    o.reset(0.4, 0.3, 20.0, clip=1)                                               # starts inside a get-up clip: getting up from its time
    g = o.getup_state()
    assert g["getting_up"] and g["timer"] == 0.4
    goal = o.record_goal()
    assert goal[3] == pytest.approx(1.0 - 0.4 / T, abs=1e-12)
    np.testing.assert_allclose(goal[:2], [math.cos(-heading_of(o.get_pose()[0])), -math.sin(-heading_of(o.get_pose()[0]))], atol=1e-12)   # target heading 0
    step_policy(o)
    root_y, head_y = o.get_pose()[0][1], o.body_state()[0][2][1]
    want = 0.2 * min(max(root_y / 1.2, 0.0), 1.0) + 0.8 * min(max(head_y / 2.0, 0.0), 1.0)
    assert o.calc_reward() == pytest.approx(want, abs=1e-12) and 0.5 < want < 1.0
    assert o.getup_state()["timer"] == pytest.approx(0.4 + 20 / 600.0, abs=1e-12)
    # throw the character down while it is "getting up": contact, but neither fallen nor terminated; once the get-up time is over it is
    rng = np.random.default_rng(1)
    st = o.action_statics()
    seen_protected = seen_fail = False
    for k in range(120):
        step_policy(o, np.clip(-st[0] + 1.0 / st[1] * rng.standard_normal(o.action_size), st[2], st[3]))
        g = o.getup_state()
        if g["contact_fall"] and g["getting_up"]:
            seen_protected = True
            assert not o.has_fallen() and o.check_terminate() == 0
        if g["contact_fall"] and not g["getting_up"]:
            seen_fail = True
            assert o.has_fallen() and o.check_terminate() == 1 and o.calc_reward() == 0.0   # heading reward of a fallen character
            break
    assert seen_protected and seen_fail
    # an episode that starts in an ordinary clip is not getting up: phase 0 and the heading reward
    o.reset(0.2, 0.0, 20.0, clip=0)
    assert not o.getup_state()["getting_up"] and o.record_goal()[3] == 0.0
    o2 = Oracle(HEADING, asset_root)
    o2.set_task_stream(2, 0, o.task_counter() - 4); o2.reset(0.2, 0.0, 20.0, clip=0)   # the reset consumed 4 draws in both scenes
    for _ in range(3):
        step_policy(o); step_policy(o2)
    assert o.calc_reward() == o2.calc_reward() and np.array_equal(o.record_goal()[:3], o2.record_goal())


def test_getup_recovery_episodes_and_test_mode_getups(asset_root):
    """ActivateRecoveryEpisode / ResetRecoveryEpisode (:40-58,301-317): after a failed episode, with probability p the fallen character is NOT
    reset -- timers and controller restart and it has to get up.  Test mode: a fall starts a get-up instead of ending the episode (:245-254)."""
    rng = np.random.default_rng(3)

    def fall(o):
        st = o.action_statics()
        for _ in range(200):
            step_policy(o, np.clip(-st[0] + 1.0 / st[1] * rng.standard_normal(o.action_size), st[2], st[3]))
            if o.is_episode_end():
                return
        raise AssertionError("the character did not fall")

    o = Oracle(["--recover_episode_prob", "1"] + GETUP, asset_root)
    o.set_task_stream(8, 3, 0)
    o.reset(0.2, 0.0, 20.0, clip=0)
    fall(o)
    assert o.check_terminate() == 1
    pose, vel = o.get_pose()
    k0, tgt = o.task_counter(), o.task_state()
    o.reset(0.5, 1.0, 7.0, clip=3)                                                 # the injected clip / time / rotation are ignored: recovery
    assert o.task_counter() == k0 + 1                                              # only the coin was drawn
    p2, v2 = o.get_pose()
    assert np.array_equal(pose, p2) and np.array_equal(vel, v2) and o.current_clip() == 0
    g = o.getup_state()
    assert g["getting_up"] and g["timer"] == 0.0 and o.record_goal()[3] == 1.0
    assert o.get_time() == 0.0 and o.need_new_action() and not o.is_episode_end() and not o.has_fallen()
    t2 = o.task_state()
    assert t2["timer_max"] == tgt["timer_max"] and np.array_equal(t2["target_pos"], tgt["target_pos"]) and np.all(t2["prev_action_com"] == 0)
    for _ in range(20):
        step_policy(o)
    assert o.get_time() == pytest.approx(20 * 20 / 600.0, abs=1e-9)               # the 7 s limit of the recovery episode is live
    # probability 0 (and test mode): ordinary reset
    o = Oracle(["--recover_episode_prob", "0"] + GETUP, asset_root)
    o.set_task_stream(8, 3, 0); o.reset(0.2, 0.0, 20.0, clip=0)
    fall(o)
    o.reset(0.5, 0.0, 20.0, clip=1)
    assert o.current_clip() == 1 and o.getup_state()["timer"] == 0.5 and not o.has_fallen()
    # test mode: the fall flips the scene into getting up and the episode goes on
    o = Oracle(GETUP, asset_root)
    o.L.dmo_set_mode(o.h, 1)
    o.set_task_stream(8, 3, 0); o.reset(0.2, 0.0, 20.0, clip=0)
    st = o.action_statics()
    began = False
    for _ in range(200):
        step_policy(o, np.clip(-st[0] + 1.0 / st[1] * rng.standard_normal(o.action_size), st[2], st[3]))
        if o.getup_state()["getting_up"]:
            began = True
            assert o.getup_state()["contact_fall"] or o.getup_state()["timer"] > 0
            assert not o.is_episode_end() and not o.has_fallen()
            break
    assert began


@pytest.mark.parametrize("clip", [2, 3])
def test_pretrained_getup_policy_stands_up_and_follows_the_heading_in_the_oracle(asset_root, clip):
    """The reference's heading + get-up policy (fp16 fixture) starts lying on the ground (get-up clips 2 / 3 of its dataset, which the
    committed archive holds in full), stands up (head above 1.3 m) and then earns the heading reward for the rest of the 20 s (0.97 measured
    over the last 10 s)."""
    a = fixture_task_actor("heading_getup")
    o = Oracle(["--arg_file", "args/train_amp_heading_getup_humanoid3d_locomotion_getup_args.txt"], asset_root)
    o.L.dmo_set_mode(o.h, 1)
    o.set_task_stream(4, 0, 0)
    o.reset(0.0, 0.4, 20.0, clip=clip)
    assert o.record_goal()[3] == 1.0 and o.body_state()[0][2][1] < 0.5            # phase 1, head near the ground
    rew, head = [], []
    for _ in range(600):
        if o.is_episode_end():
            break
        o.set_action(gated_actor_mode(a, o.record_state(), o.record_goal()))
        for _ in range(20):
            o.update(1.0 / 600.0)
        rew.append(o.calc_reward()); head.append(o.body_state()[0][2][1])
    assert len(rew) == 600 and not o.has_fallen()
    assert max(head) > 1.3 and head[-1] > 1.25 and np.mean(rew[300:]) > 0.85, (max(head), head[-1], np.mean(rew[300:]))


# ------------------------------------------------------------------------------------------------ strike_amp (cSceneStrikeAMP)
STRIKE = ["--scene", "strike_amp", "--target_hit_reset_time", "2", "--target_radius", "0.2", "--target_min", "-0.5", "1.2", "0.6", "--target_max", "0.5", "1.4", "1.1",
          "--tar_near_dist", "1.4", "--tar_far_prob", "0.4", "--strike_bodies", "8", "--fail_tar_contact_bodies", "0", "1", "2", "--init_hit_prob", "0.1",
          "--hit_tar_speed", "1.5", "--tar_reward_scale", "2"] + TARGET


def test_strike_reset_draw_order_goal_and_rewards(asset_root):
    """SceneStrikeAMP.cpp: reset draws (:300-383), goal = target in the origin frame + hit phase (:407-430), train reward in its three regimes
    (:22-190), hit detection (:440-481), forbidden-body failure and success after the hold time (:489-546)."""
    o = Oracle(STRIKE, asset_root)
    assert o.goal_size == 4 and o.enable_amp_task_reward()
    o.set_task_stream(13, 2, 0)
    o.reset(0.3, 0.0, 20.0, clip=0)
    s = Stream(13, 2)
    s.uniform(5.0, 10.0)                                                         # target timer (--rand_target_time_min/max of the target args)
    far = s.coin(0.4)
    theta = s.uniform(-math.pi, math.pi) if far else s.uniform(-0.5, 0.5)
    h = s.uniform(1.2, 1.4)
    dist = s.uniform(0.6, 10.0) if far else s.uniform(0.6, 1.1)
    hit0 = s.coin(0.1)                                                           # ResetTargetHit (train mode, init_hit_prob 0.1)
    hit_time = s.uniform(0.0 - 2.0, 0.0) if hit0 else -1.0
    root = o.get_pose()[0][:3]
    ts, ss = o.task_state(), o.strike_state()
    np.testing.assert_allclose([ts["target_pos"][0], ss["target_height"], ts["target_pos"][2]],
                               [root[0] + dist * math.cos(theta), h, root[2] - dist * math.sin(theta)], atol=1e-7)
    assert ss["hit"] == hit0 and ss["hit_time"] == pytest.approx(hit_time, abs=1e-12) and o.task_counter() == s.k
    step_policy(o); step_policy(o)
    pose = o.get_pose()[0]
    root, hd = pose[:3], heading_of(pose)
    pos, rot, lv, av = o.body_state()
    com = com_of(o, asset_root)
    ts = o.task_state()
    c, s_ = math.cos(-hd), math.sin(-hd)

    def put_target(p, hit=False, hit_time=-1.0):
        o.set_task_state(p, 1.0, 0.0, ts["timer"], ts["timer_max"], ts["prev_action_com"])
        o.set_strike_state(hit, hit_time)

    hand = pos[8]
    # far regime: 0.3 * (0.7 exp(-0.5 max(d - 1.4, 0)^2) + 0.3 vel term)
    tar = np.array([root[0] + 4.0, 1.3, root[2] + 1.0])
    put_target(tar)
    d = math.hypot(tar[0] - root[0], tar[2] - root[2])
    cd = np.array([tar[0] - com[0], 0.0, tar[2] - com[2]]); cd /= np.linalg.norm(cd)
    avg = float(cd @ (com - ts["prev_action_com"])) / (19 / 600.0)
    vel_r = 0.0 if avg < 0 else math.exp(-4.0 * max(1.0 - avg, 0.0) ** 2)
    assert o.calc_reward() == pytest.approx(0.3 * (0.7 * math.exp(-0.5 * (d - 1.4) ** 2) + 0.3 * vel_r), abs=1e-9)
    loc = np.array([tar[0] - root[0], tar[1], tar[2] - root[2]])
    np.testing.assert_allclose(o.record_goal(), [c * loc[0] + s_ * loc[2], loc[1], -s_ * loc[0] + c * loc[2], 0.0], atol=1e-9)
    # near regime: 0.3 + 0.3 * max over strike bodies of (0.2 exp(-2 |t - hand|^2) + 0.8 clamp(v.dir / 1.5)^2)
    tar = hand + np.array([0.25, 0.05, -0.1])
    put_target(tar)
    dirn = np.array([tar[0] - root[0], 0.0, tar[2] - root[2]]); dirn /= np.linalg.norm(dirn)
    near = 0.2 * math.exp(-2.0 * float(((tar - hand) ** 2).sum())) + 0.8 * min(max(float(dirn @ lv[8]) / 1.5, 0.0), 1.0) ** 2
    assert o.calc_reward() == pytest.approx(0.3 + 0.3 * near, abs=1e-9) and o.check_terminate() == 0
    # hit: full reward, phase grows with the hold time, success (terminate 2) once it reaches the reset time
    t_now = o.get_time()
    put_target(tar, hit=True, hit_time=t_now - 0.5)
    assert o.calc_reward() == pytest.approx(1.0, abs=1e-12) and o.record_goal()[3] == pytest.approx(0.25, abs=1e-12) and o.check_terminate() == 0
    put_target(tar, hit=True, hit_time=t_now - 2.0)
    assert o.record_goal()[3] == 1.0 and o.check_terminate() == 2 and o.is_episode_end()
    # a forbidden body (root / torso / head) at the target fails the episode; too far fails it as well
    put_target(pos[1] + np.array([0.05, 0.0, 0.05]))
    assert o.check_terminate() == 1
    put_target(np.array([root[0] + 15.5, 1.3, root[2]]))
    assert o.check_terminate() == 1
    # hit detection needs both the hand inside the sphere and enough speed towards the target: standing still near it is no hit
    put_target(hand + np.array([0.05, 0.0, 0.0]))
    o.update(1.0 / 600.0)
    assert not o.strike_state()["hit"]


@needs_reference
@pytest.mark.parametrize("seed,far", [(1, False), (7, True)])
def test_pretrained_strike_policy_punches_the_target_in_the_oracle(seed, far):
    """The reference's walk-and-punch policy hits the oracle-drawn target with its hand (fast enough, from the right side) and holds for the 2 s
    that make the episode a success (terminate code 2) -- also when it first has to walk 5 m to get there."""
    from deepmimic_b200.tf_checkpoint import load_actor
    ref = reference_root()
    a = _f64(load_actor(os.path.join(ref, "data/policies/humanoid3d_amp/humanoid3d_amp_strike_walk_punch.ckpt")))
    o = Oracle(["--arg_file", "args/run_amp_strike_humanoid3d_walk_punch_args.txt"], ref)
    o.L.dmo_set_mode(o.h, 1)
    o.set_task_stream(seed, 0, 0)
    o.reset(0.3, 0.0, 20.0, clip=0)
    tp, root = o.task_state()["target_pos"], o.get_pose()[0]
    assert (math.hypot(tp[0] - root[0], tp[2] - root[2]) > 3.0) == far
    hit_step = None
    for k in range(600):
        if o.is_episode_end():
            break
        o.set_action(gated_actor_mode(a, o.record_state(), o.record_goal()))
        for _ in range(20):
            o.update(1.0 / 600.0)
            if o.is_episode_end():
                break
        if hit_step is None and o.strike_state()["hit"]:
            hit_step = k
    assert hit_step is not None and o.check_terminate() == 2 and not o.has_fallen(), (hit_step, o.check_terminate())
    assert o.get_time() == pytest.approx((hit_step + 1) / 30.0 + 2.0, abs=0.05)     # success exactly the hold time after the hit


# ------------------------------------------------------------------------------------------------ dm_task_ext.cuh on the host (get-up, strike)
def _ext_params(getup_time=0.0, root_h=0.5, head_h=0.5, recover=0.0, head_id=0, strike=(), fail=(), init_hit=0.0):
    q = np.zeros(32)
    q[0:4] = [getup_time, root_h, head_h, recover]
    q[4:7] = [-0.5, 1.2, 0.6]; q[7:10] = [0.5, 1.4, 1.1]
    q[10:17] = [0.2, 2.0, 2.0, 1.5, init_hit, 0.4, 1.4]
    q[17] = head_id; q[18] = len(strike); q[19:19 + len(strike)] = strike; q[23] = len(fail); q[24:24 + len(fail)] = fail
    return q


def _task_params(kind, timer=(1.0, 5.0), max_dist=10.0, succ=0.5, fail=15.0, pos_scale=0.5, tar_speed=1.0, min_vel=1):
    p = np.zeros(16)
    p[0:7] = [kind, timer[0], timer[1], max_dist, succ, fail, pos_scale]
    p[7:13] = [0.15, 0.01, 0.02, 1.0, 5.0, 0.25]
    p[13], p[14] = tar_speed, min_vel
    return p


def _bodies(o, xq):
    pos, rot, lv, av = o.body_state()
    b = np.zeros(38)
    b[0] = pos[int(xq[17])][1]; b[1] = float(o.getup_state()["contact_fall"])
    for k in range(int(xq[18])):
        b[2 + 3 * k: 5 + 3 * k] = pos[int(xq[19 + k])]; b[14 + 3 * k: 17 + 3 * k] = lv[int(xq[19 + k])]
    for k in range(int(xq[23])):
        b[26 + 3 * k: 29 + 3 * k] = pos[int(xq[24 + k])]
    return b


def _shim_ext_signatures(L):
    import ctypes as C
    d, dp_, u64, i = C.c_double, C.POINTER(C.c_double), C.c_uint64, C.c_int
    L.shim_getup_reset.argtypes = [dp_, dp_, d, i]
    L.shim_getup_try_recovery.argtypes = [dp_, dp_, u64, u64, i, i]
    L.shim_getup_recovery_reset.argtypes = [dp_, dp_]
    L.shim_getup_update.argtypes = [dp_, dp_, d, i, i]
    L.shim_getup_phase.argtypes = [dp_, dp_]; L.shim_getup_phase.restype = d
    L.shim_getup_reward.argtypes = [dp_, d, d]; L.shim_getup_reward.restype = d
    L.shim_strike_reset.argtypes = [dp_, dp_, dp_, dp_, u64, u64, d, d, d, i]
    L.shim_strike_update.argtypes = [dp_, dp_, dp_, dp_, u64, u64, d, d, d, d, dp_]
    L.shim_strike_terminate.argtypes = [dp_, dp_, dp_, dp_, d, d, d]
    L.shim_strike_goal.argtypes = [dp_, dp_, dp_, d, d, d, d, dp_]
    L.shim_strike_reward.argtypes = [dp_, dp_, dp_, dp_, i, d, d, d, i, i, d, d]; L.shim_strike_reward.restype = d
    return L


def test_device_strike_logic_matches_the_oracle_on_the_host(asset_root, task_shim):
    """dm_task_ext.cuh (host build) against the oracle's strike scene over 5 s of a random policy, with the target re-placed in front of the moving
    hand every second so that hits, holds, successes and forbidden-body failures all occur: hit state / time, goal, reward and termination code
    after every update."""
    L = _shim_ext_signatures(task_shim)
    o = Oracle(STRIKE, asset_root)
    P, X = _task_params(1, timer=(5.0, 10.0)), _ext_params(head_id=2, strike=(8,), fail=(0, 1, 2), init_hit=0.1)   # STRIKE sits on the target args: timer 5..10 s
    seed, env = 5, 9
    o.set_task_stream(seed, env, 0)
    o.reset(0.3, 0.0, 20.0, clip=0)
    t, x = np.zeros(16), np.zeros(8)
    root = o.get_pose()[0]
    L.shim_strike_reset(_ptr(P), _ptr(X), _ptr(t), _ptr(x), seed, env, root[0], root[2], 0.0, 0)
    rng = np.random.default_rng(0)
    st = o.action_statics()
    seen = dict(hit=0, succ=0, fail=0, near=0, far=0)

    def compare(k):
        ts, ss = o.task_state(), o.strike_state()
        np.testing.assert_allclose([t[0], x[0], t[1]], [ts["target_pos"][0], ss["target_height"], ts["target_pos"][2]], atol=1e-7)
        assert bool(x[1]) == ss["hit"] and x[2] == pytest.approx(ss["hit_time"], abs=1e-12), k
        assert t[4] == pytest.approx(ts["timer"], abs=1e-12) and t[5] == pytest.approx(ts["timer_max"], rel=1e-15) and int(t[12]) == o.task_counter()
    compare(-1)
    for k in range(3000):
        if k == 1:              # first second: a far target (the far regime of the reward)
            rp = o.get_pose()[0]
            tar = np.array([rp[0] + 5.0, 1.3, rp[2] + 1.0])
            ts = o.task_state()
            o.set_task_state(tar, 1.0, 0.0, ts["timer"], ts["timer_max"], ts["prev_action_com"]); o.set_strike_state(False, -1.0)
            t[0], x[0], t[1] = tar[0], tar[1], tar[2]; x[1], x[2] = 0.0, -1.0
        if k in (301, 2101):    # (between two action boundaries) the target goes where the hand will be -- hit, 2 s hold, success -- and later onto the chest (forbidden)
            pos, _, lv, _ = o.body_state()
            tar = pos[8] + 0.02 * lv[8] / (np.linalg.norm(lv[8]) + 1e-9) if k == 301 else pos[1] + np.array([0.0, 0.05, 0.0])
            ts = o.task_state()
            o.set_task_state(tar, 1.0, 0.0, ts["timer"], ts["timer_max"], ts["prev_action_com"]); o.set_strike_state(False, -1.0)
            t[0], x[0], t[1] = tar[0], tar[1], tar[2]; x[1], x[2] = 0.0, -1.0
        if o.need_new_action():
            ts = o.task_state(); t[6:9] = ts["prev_action_com"]; t[9:12] = o.calc_com()
            pose = o.get_pose()[0]
            g = np.zeros(4)
            L.shim_strike_goal(_ptr(X), _ptr(t), _ptr(x), pose[0], pose[2], heading_of(pose), o.get_time(), _ptr(g))
            np.testing.assert_allclose(g, o.record_goal(), atol=1e-9)
            if k > 0:
                r = L.shim_strike_reward(_ptr(P), _ptr(X), _ptr(t), _ptr(x), int(o.has_fallen()), pose[0], pose[2], 19.0 / 600.0, 0, o.check_terminate(), 20.0, o.get_time())
                assert r == pytest.approx(o.calc_reward(), abs=1e-9), k
                d = math.hypot(t[0] - pose[0], t[1] - pose[2])
                seen["near" if d < 1.4 else "far"] += 1
            o.set_action(np.clip(-st[0] + 0.3 / st[1] * rng.standard_normal(o.action_size), st[2], st[3]))
        o.update(1.0 / 600.0)
        root = o.get_pose()[0]
        L.shim_strike_update(_ptr(P), _ptr(X), _ptr(t), _ptr(x), seed, env, 1.0 / 600.0, root[0], root[2], o.get_time(), _ptr(_bodies(o, X)))
        compare(k)
        code = L.shim_strike_terminate(_ptr(P), _ptr(X), _ptr(t), _ptr(x), root[0], root[2], o.get_time())
        if not o.has_fallen():
            assert code == o.check_terminate(), k
        seen["hit"] += int(x[1]); seen["succ"] += int(code == 2); seen["fail"] += int(code == 1)
    assert min(seen.values()) > 0, seen


def test_device_getup_logic_matches_the_oracle_on_the_host(asset_root, task_shim):
    """dm_task_ext.cuh's get-up pieces against the oracle: timer / phase / reward through a reset in a get-up clip, a fall, a recovery episode
    (train mode) and a test-mode get-up."""
    L = _shim_ext_signatures(task_shim)
    rng = np.random.default_rng(4)
    for mode in (0, 1):
        o = Oracle(["--recover_episode_prob", "1"] + GETUP, asset_root)
        o.L.dmo_set_mode(o.h, mode)
        dur = o.clip_table()[0]
        X = _ext_params(getup_time=max(dur[1], dur[2]), root_h=1.2, head_h=2.0, recover=1.0, head_id=2)
        seed, env = 6, 1
        o.set_task_stream(seed, env, 0)
        o.reset(0.4, 0.0, 20.0, clip=1)
        t, x = np.zeros(16), np.zeros(8)
        L.shim_getup_reset(_ptr(X), _ptr(x), 0.4, 1)
        st = o.action_statics()
        recoveries = began = 0
        for k in range(2400):
            if o.is_episode_end():
                assert mode == 0                                                   # test mode never ends on a fall here: it gets up instead
                t[12] = o.task_counter()
                rec = L.shim_getup_try_recovery(_ptr(X), _ptr(t), seed, env, mode, o.check_terminate())
                o.reset(0.2, 0.0, 20.0, clip=0)
                assert int(t[12]) == o.task_counter() - (0 if rec else 4)         # a full reset also draws timer, target x2 and speed
                if rec:
                    L.shim_getup_recovery_reset(_ptr(t), _ptr(x)); recoveries += 1
                else:
                    L.shim_getup_reset(_ptr(X), _ptr(x), 0.2, 0)
                if recoveries >= 2:
                    break
            if o.need_new_action():
                g = o.getup_state()
                assert L.shim_getup_phase(_ptr(X), _ptr(x)) == pytest.approx(o.record_goal()[3], abs=1e-12)
                if g["getting_up"]:
                    assert L.shim_getup_reward(_ptr(X), o.get_pose()[0][1], o.body_state()[0][2][1]) == pytest.approx(o.calc_reward(), abs=1e-7)   # root height through the float link frames in the oracle
                o.set_action(np.clip(-st[0] + 1.0 / st[1] * rng.standard_normal(o.action_size), st[2], st[3]))
            before = o.getup_state()["getting_up"]
            o.update(1.0 / 600.0)
            g = o.getup_state()
            up = L.shim_getup_update(_ptr(X), _ptr(x), 1.0 / 600.0, mode, int(g["contact_fall"]))
            assert bool(up) == g["getting_up"] and x[3] == pytest.approx(g["timer"], abs=1e-12), k
            began += int(g["getting_up"] and not before)
        assert (recoveries >= 2) if mode == 0 else (began >= 1)


def test_fixture_getup_and_strike_policies_in_the_oracle_without_the_reference_tree(asset_root):
    """Hermetic pins for the two other task scenes on the committed assets: the get-up policy (real get-up clips, shipped in the archive) stands
    up from lying face down and then follows the heading; the strike policy, reset from the mini dataset, walks to a far target and punches it."""
    a = fixture_task_actor("heading_getup")
    o = Oracle(["--arg_file", "args/train_amp_heading_getup_humanoid3d_locomotion_getup_args.txt"], asset_root)
    o.L.dmo_set_mode(o.h, 1)
    o.set_task_stream(4, 0, 0)
    o.reset(0.0, 0.4, 20.0, clip=2)
    assert o.num_clips() == 4 and o.record_goal()[3] == 1.0 and o.body_state()[0][2][1] < 0.5
    rew, head = [], []
    for _ in range(600):
        o.set_action(gated_actor_mode(a, o.record_state(), o.record_goal()))
        for _ in range(20):
            o.update(1.0 / 600.0)
        rew.append(o.calc_reward()); head.append(o.body_state()[0][2][1])
    assert not o.is_episode_end() or o.get_time() >= 20.0 - 1e-6
    assert not o.has_fallen() and max(head) > 1.3 and np.mean(rew[300:]) > 0.85, (max(head), np.mean(rew[300:]))
    a = fixture_task_actor("strike")
    o = Oracle(MINI + ["--arg_file", "args/train_amp_strike_humanoid3d_walk_punch_args.txt"], asset_root)
    o.L.dmo_set_mode(o.h, 1)
    for seed in range(1, 40):                                                  # a seed whose first target is a far one
        o.set_task_stream(seed, 0, 0)
        o.reset(0.3, 0.0, 20.0, clip=1)
        tp, root = o.task_state()["target_pos"], o.get_pose()[0]
        if math.hypot(tp[0] - root[0], tp[2] - root[2]) > 3.0:
            break
    hit = None
    for k in range(600):
        if o.is_episode_end():
            break
        o.set_action(gated_actor_mode(a, o.record_state(), o.record_goal()))
        for _ in range(20):
            o.update(1.0 / 600.0)
            if o.is_episode_end():
                break
        if hit is None and o.strike_state()["hit"]:
            hit = k
    assert hit is not None and o.check_terminate() == 2 and not o.has_fallen(), (hit, o.check_terminate())
