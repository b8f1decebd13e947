"""Known-answer tests that pin the CPU oracle WITHOUT Bullet (SURVEY.md 8(c)): the reference ships no tests or golden
vectors, so these are derived from the reference's own semantics.  CPU only."""
import json
import os

import numpy as np
import pytest

from deepmimic_b200.assets import reference_root
from tests.oracle_binding import Oracle

SPINKICK = ["--arg_file", "args/run_humanoid3d_spinkick_args.txt"]
WALK = ["--arg_file", "args/train_humanoid3d_walk_args.txt"]
DOG = ["--arg_file", "args/train_dog3d_trot_args.txt"]


def _layout(asset_root, char_file):
    d = json.load(open(os.path.join(asset_root, char_file)))
    types = [j["Type"] for j in d["Skeleton"]["Joints"]]
    off, o = [], 0
    for i, t in enumerate(types):
        off.append(o)
        o += 7 if i == 0 else {"spherical": 4, "revolute": 1, "fixed": 0}[t]
    return types, off, o


@pytest.mark.parametrize("args,nj,pose,dofs,state,action", [(SPINKICK, 15, 43, 34, 227, 28), (DOG, 23, 83, 64, 347, 58)])
def test_dims(asset_root, args, nj, pose, dofs, state, action):
    o = Oracle(args, asset_root)
    assert (o.num_joints, o.pose_dim, o.num_dofs, o.state_size, o.action_size) == (nj, pose, dofs, state, action)


def test_motion_duration_and_frames(asset_root):
    o = Oracle(SPINKICK, asset_root)
    assert abs(o.motion_duration - 1.283282) < 1e-9 and o.num_frames == 78
    d = json.load(open(os.path.join(asset_root, "data/motions/humanoid3d_spinkick.txt")))
    fr = np.array(d["Frames"])
    times = np.concatenate([[0.0], np.cumsum(fr[:-1, 0])])
    for i in (0, 1, 17, 40, 76):
        p, _ = o.kin_frame(times[i] + 1e-12)   # the reset leaves origin at the sim root: compare joint slots only
        q = fr[i, 1 + 7:]
        for a in range(7, 43):
            pass
        # spherical quaternions are normalised at load; compare up to normalisation
        assert np.abs(p[7:] - fr[i, 8:] / 1.0).max() < 1e-5
    # cyclic: pose(t + dur) == pose(t) + root cycle delta (y zeroed)
    o.reset(0.0, 0.0, 20.0)
    p0, v0 = o.kin_frame(0.37)
    p1, v1 = o.kin_frame(0.37 + o.motion_duration)
    delta = fr[-1, 1:4] - fr[0, 1:4]
    assert np.abs((p1[:3] - p0[:3]) - np.array([delta[0], 0.0, delta[2]])).max() < 1e-9
    assert np.abs(p1[3:] - p0[3:]).max() < 1e-9 and np.abs(v1 - v0).max() < 1e-9


def test_reward_is_one_after_reset_without_ground_lift(asset_root):
    o = Oracle(SPINKICK, asset_root)
    for t0 in (0.6, 0.75, 0.9):
        o.reset(t0, 0.0, 20.0)
        r, e = o.reward_terms()
        assert abs(r - 1.0) < 1e-9, (t0, r, e)
    # when ResolveCharGroundIntersect lifts the character the kinematic origin moves with it and the reference's
    # ground-relative heights no longer agree: the deficit is exactly 4 end effectors + root, all with the same dy
    o.reset(0.0, 0.0, 20.0)
    r, e = o.reward_terms()
    assert e[0] == 0 and e[1] == 0 and abs(e[2] - 4 * e[3]) < 1e-9


def test_record_state_layout(asset_root):
    o = Oracle(SPINKICK, asset_root)
    o.reset(0.5, 0.0, 20.0)
    s = o.record_state()
    assert s.shape == (227,) and not np.isnan(s).any()
    assert abs(s[0] - np.fmod(0.5 / o.motion_duration, 1.0)) < 1e-12       # phase slot
    p, _ = o.get_pose()
    assert abs(s[1] - p[1]) < 1e-6                                          # root height
    nrm = s[2 + 3:2 + 6]; tan = s[2 + 6:2 + 9]
    assert abs(np.linalg.norm(nrm) - 1) < 1e-6 and abs(np.linalg.norm(tan) - 1) < 1e-6 and abs(nrm @ tan) < 1e-6


@pytest.mark.parametrize("args,char,mass", [(SPINKICK, "data/characters/humanoid3d.txt", 45.0), (DOG, "data/characters/dog3d.txt", 29.25)])
def test_crba_rnea_self_consistency(asset_root, args, char, mass):
    o = Oracle(args, asset_root)
    types, off, n = _layout(asset_root, char)
    o.reset(0.3, 0.0, 20.0)
    rng = np.random.default_rng(0)
    p, v = o.get_pose()
    v = rng.standard_normal(n)
    v[6] = 0
    for j, t in enumerate(types):
        if t == "spherical":
            v[off[j] + 3] = 0
    o.set_pose_vel(p, v)
    M, Cb = o.rbd_mass_bias()
    assert abs(M[0, 0] - mass) < 1e-9 and abs(M[1, 1] - mass) < 1e-9          # total mass
    assert np.abs(M - M.T).max() < 1e-12
    live = [i for i in range(n) if M[i, i] != 0]
    assert len(live) == o.num_dofs
    assert np.linalg.eigvalsh(M[np.ix_(live, live)]).min() > 0
    acc = rng.standard_normal(n)
    acc[[i for i in range(n) if i not in live]] = 0
    tau = o.inv_dyna(acc)
    assert np.abs(tau - (M @ acc + Cb)).max() < 1e-9                          # SolveInvDyna(acc) == M acc + C
    # C(q, 0) is the gravity generalised force: linear root rows carry -m g
    o.set_pose_vel(p, np.zeros(n))
    _, Cg = o.rbd_mass_bias()
    assert np.abs(Cg[:3] - np.array([0, mass * 9.8, 0])).max() < 1e-9


def test_spd_fixed_point(asset_root):
    """target == current pose, zero velocity: SPD torque equals the PD term of the gravity-induced motion only;
    with the action set to the current pose and zero gains on the root the torque stays bounded and finite."""
    o = Oracle(SPINKICK, asset_root)
    o.reset(0.2, 0.0, 20.0)
    tau = o.spd_tau(1.0 / 600.0)
    assert np.isfinite(tau).all() and np.abs(tau[:7]).max() == 0.0


def test_need_new_action_every_20_updates(asset_root):
    o = Oracle(SPINKICK, asset_root)
    for t0 in (0.0, 0.777):
        o.reset(t0, 0.0, 100.0)
        assert o.need_new_action()
        hits = []
        for k in range(1, 101):
            o.set_action(np.zeros(o.action_size)) if o.need_new_action() else None
            o.update(1.0 / 600.0)
            if o.need_new_action():
                hits.append(k)
            if o.is_episode_end():
                break
        assert hits[:4] == [20, 40, 60, 80][:len(hits[:4])]


def test_action_tables(asset_root):
    o = Oracle(SPINKICK, asset_root)
    off, scl, lo, hi = o.action_statics()
    # spherical: bounds +-2pi, scale 1/pi, offset 0 ; knee (revolute [-3.14, 0]): offset 1.57, scale 1/6.28, bounds mean +- 2*range
    assert np.allclose(lo[:3], -2 * np.pi) and np.allclose(hi[:3], 2 * np.pi) and np.allclose(scl[:3], 1 / np.pi) and np.allclose(off[:3], 0)
    knee = 3 + 3 + 3
    assert abs(off[knee] - 1.57) < 1e-12 and abs(scl[knee] - 0.5 / 3.14) < 1e-12 and abs(lo[knee] - (-1.57 - 6.28)) < 1e-12 and abs(hi[knee] - (-1.57 + 6.28)) < 1e-12


def _box_character_root(asset_root, tmp_path):
    """copy of humanoid3d whose capsules are replaced by boxes: DeepMimic's exact-shape inertia and Bullet's
    collision-shape inertia then coincide, so the restated Bullet ABA must equal DeepMimic's M^-1 (tau - C)."""
    root = tmp_path / "assets"
    (root / "data" / "characters").mkdir(parents=True)
    (root / "args").mkdir()
    for sub in ("controllers", "motions", "terrain"):
        os.symlink(os.path.join(asset_root, "data", sub), root / "data" / sub)
    d = json.load(open(os.path.join(asset_root, "data/characters/humanoid3d.txt")))
    for b in d["BodyDefs"]:
        if b["Shape"] == "capsule":
            r, h = b["Param0"], b["Param1"]
            b["Shape"] = "box"; b["Param0"] = r; b["Param1"] = h + r; b["Param2"] = r
    d.pop("DrawShapeDefs", None)
    json.dump(d, open(root / "data" / "characters" / "box_humanoid3d.txt", "w"))
    a = open(os.path.join(asset_root, "args/run_humanoid3d_spinkick_args.txt")).read().replace("humanoid3d.txt", "box_humanoid3d.txt")
    open(root / "args" / "box_args.txt", "w").write(a)
    return str(root)


def test_bullet_aba_matches_deepmimic_rbd_on_box_character(asset_root, tmp_path):
    root = _box_character_root(asset_root, tmp_path)
    o = Oracle(["--arg_file", "args/box_args.txt"], root)
    types, off, n = _layout(asset_root, "data/characters/humanoid3d.txt")
    rng = np.random.default_rng(1)
    o.reset(0.4, 0.0, 20.0)
    p, _ = o.get_pose()
    p[1] += 1.0
    v = rng.standard_normal(n)
    v[3:7] = 0   # zero root angular velocity: the reference's root "cj" term mixes frames otherwise (see next test)
    for j, t in enumerate(types):
        if t == "spherical":
            v[off[j] + 3] = 0
    o.set_pose_vel(p, v)
    M, Cb = o.rbd_mass_bias()
    tau = rng.standard_normal(n) * 20
    tau[:7] = 0
    for j, t in enumerate(types):
        if t == "spherical":
            tau[off[j] + 3] = 0
    live = [i for i in range(n) if M[i, i] != 0]
    acc = np.zeros(n)
    acc[live] = np.linalg.solve(M[np.ix_(live, live)], (tau - Cb)[live])
    jt = []
    for j, t in enumerate(types):
        if t == "spherical":
            jt += list(16 * tau[off[j]:off[j] + 3])
        elif t == "revolute":
            jt += [16 * tau[off[j]]]
    out = o.bullet_aba(np.array(jt), True)
    b = [out[3] / 4, out[4] / 4, out[5] / 4, out[0], out[1], out[2], 0]
    k = 6
    for j, t in enumerate(types):
        if t == "spherical":
            b += list(out[k:k + 3]) + [0]; k += 3
        elif t == "revolute":
            b += [out[k]]; k += 1
    b = np.array(b)
    assert np.abs(acc - b).max() / np.abs(acc).max() < 2e-6


def test_reference_root_cj_quirk_is_restated(asset_root, tmp_path):
    """cRBDUtil::BuildCjRoot differentiates the root quaternion with the body-frame formula applied to the WORLD angular
    velocity (RBDUtil.cpp:915-958); the oracle restates that literally, so with a spinning, translating root its linear
    root acceleration differs from rigid-body truth (the Bullet-side ABA) while every joint acceleration still agrees."""
    root = _box_character_root(asset_root, tmp_path)
    o = Oracle(["--arg_file", "args/box_args.txt"], root)
    types, off, n = _layout(asset_root, "data/characters/humanoid3d.txt")
    o.reset(0.4, 0.0, 20.0)
    p, _ = o.get_pose()
    p[1] += 1.0
    v = np.zeros(n); v[0:3] = [1.0, 0.5, -2.0]; v[3:6] = [0.7, -1.1, 0.4]
    o.set_pose_vel(p, v)
    M, Cb = o.rbd_mass_bias()
    live = [i for i in range(n) if M[i, i] != 0]
    acc = np.zeros(n); acc[live] = np.linalg.solve(M[np.ix_(live, live)], (-Cb)[live])
    out = o.bullet_aba(np.zeros(o.num_dofs - 6), True)
    assert np.abs(acc[3:6] - out[0:3]).max() < 1e-3          # angular root acceleration agrees
    assert np.abs(acc[0:3] - out[3:6] / 4).max() > 0.1       # linear one does not: the quirk


def test_free_fall_com_acceleration_is_g(asset_root):
    o = Oracle(SPINKICK, asset_root)
    o.reset(0.3, 0.0, 20.0)
    p, v = o.get_pose()
    p[1] += 2.0
    o.set_pose_vel(p, np.zeros_like(v))
    out = o.bullet_aba(np.zeros(o.num_dofs - 6), True)
    # zero velocity, no torques: every point of the character accelerates at g (scaled units x4)
    assert np.abs(out[3:6] - np.array([0, -9.8 * 4, 0])).max() < 2e-3 and np.abs(out[:3]).max() < 2e-3 and np.abs(out[6:]).max() < 5e-3


def make_short_nonlooping_clip(asset_root, tmp_path, frames=6):
    """The first `frames` frames of the walk clip with "Loop": "none" (the shipped test assets only hold looping clips)."""
    import json
    src = json.load(open(os.path.join(asset_root, "data/motions/humanoid3d_walk.txt")))
    clip = {"Loop": "none", "Frames": src["Frames"][:frames]}
    path = os.path.join(str(tmp_path), "short_nonlooping.txt")
    json.dump(clip, open(path, "w"))
    return path, sum(f[0] for f in clip["Frames"][:-1])


def test_finished_clip_fails_the_episode_in_imitate_only(asset_root, tmp_path):
    """cSceneImitate::CheckTerminate adds cMotion::IsOver (SceneImitate.cpp:193-205, Motion.cpp:529-532); the AMP scenes use
    cRLSceneSimChar::CheckTerminate alone (SceneImitateAMP.cpp:185-189)."""
    clip, dur = make_short_nonlooping_clip(asset_root, tmp_path)
    res = {}
    for scene in ("imitate", "imitate_amp"):
        o = Oracle(["--scene", scene, "--motion_file", clip, "--arg_file", "args/train_humanoid3d_walk_args.txt"], asset_root)
        o.reset(0.0, 0.0, 20.0)
        n = int(np.ceil(dur * 600.0)) + 2
        hist = []
        for i in range(n):
            o.update(1.0 / 600.0)
            hist.append((o.check_terminate(), o.is_episode_end(), o.has_fallen()))
        res[scene] = hist
        assert not any(h[2] for h in hist)                      # nobody falls in 0.2 s
    k = int(np.floor(dur * 600.0)) - 2
    assert all(h[0] == 0 for h in res["imitate"][:k]) and res["imitate"][-1][0] == 1 and res["imitate"][-1][1]
    assert all(h[0] == 0 and not h[1] for h in res["imitate_amp"])


def test_root_rotation_sync_rotates_the_kinematic_origin(asset_root):
    """--sync_char_root_rot true (dog3d_spin): SyncKinCharRoot / SyncKinCharNewCycle call RotateRoot, whose virtual SetRootRotation lands in
    cKinCharacter::RotateOrigin (SceneImitate.cpp:386-444, Character.cpp:210-216, KinCharacter.cpp:243-248,285-327): the heading difference
    becomes part of the ORIGIN rotation and persists over the following updates."""
    def heading(q):   # pose quaternion (w, x, y, z): cKinTree::CalcHeading
        w, x, y, z = q
        return np.arctan2(-(2 * (x * z - w * y)), 1 - 2 * (y * y + z * z))
    o = Oracle(["--sync_char_root_rot", "true", "--arg_file", "args/train_humanoid3d_walk_args.txt"], asset_root)
    o.reset(0.2, 0.0, 20.0)
    nj = o.num_joints
    origin_rot = lambda: o.get_snapshot()[13 + 55 * nj + 4: 13 + 55 * nj + 8]
    np.testing.assert_allclose(origin_rot(), [1, 0, 0, 0], atol=1e-8)           # sim was just synced to the clip (through float state): nothing to rotate
    # turn the simulated character by 0.7 rad about +y and run through the end of the cycle with the default PD targets
    p, v = o.get_pose()
    c, s_ = np.cos(0.35), np.sin(0.35)
    w, x, y, z = p[3:7]
    p[3:7] = [c * w - s_ * y, c * x + s_ * z, c * y + s_ * w, c * z - s_ * x]    # (c, 0, s, 0) * q
    o.set_pose_vel(p, v)
    dur = o.motion_duration
    n = int(np.ceil((dur - 0.2) * 600.0)) + 1
    for _ in range(n):
        o.update(1.0 / 600.0)
    q = origin_rot()
    assert abs(2 * np.arctan2(q[2], q[0])) > 0.3                                  # the origin picked up (most of) the turn ...
    kin, sim = o.get_kin_pose()[0], o.get_pose()[0]
    for _ in range(30):                                                           # ... and keeps it: no snap back on the next updates
        o.update(1.0 / 600.0)
    np.testing.assert_allclose(origin_rot(), q, atol=1e-12)
    # right after the wrap the two headings agreed
    o2 = Oracle(["--sync_char_root_rot", "true", "--arg_file", "args/train_humanoid3d_walk_args.txt"], asset_root)
    o2.reset(0.2, 0.0, 20.0)
    o2.set_pose_vel(p, v)
    prev = 0.0
    for k in range(n + 5):
        o2.update(1.0 / 600.0)
        ph = (0.2 + (k + 1) / 600.0) / dur % 1.0
        if ph < prev:
            assert abs(heading(o2.get_kin_pose()[0][3:7]) - heading(o2.get_pose()[0][3:7])) < 2e-2   # one update of motion apart
            break
        prev = ph
    else:
        raise AssertionError("no cycle wrap seen")


def test_amp_observation_known_answers(asset_root):
    """cSceneImitateAMP::BuildAMPObs (SceneImitateAMP.cpp:279-397): layout [pose now | pose prev | vel now | vel prev]; humanoid
    (1 + 6 + 8*6 + 4 + 4*3) = 71 and (6 + 36) = 42 -> 226 (SURVEY 8a)."""
    o = Oracle(SPINKICK, asset_root)
    assert o.amp_obs_size() == 226
    d = Oracle(DOG, asset_root)
    assert d.amp_obs_size() == 2 * ((1 + 6 + 18 * 6 + 4 + 4 * 3) + (6 + 83 - 7))
    t0 = 0.6
    o.reset(t0, 0.0, 20.0)
    a = o.record_amp_obs_agent()
    e = o.record_amp_obs_expert(t0)
    assert np.isfinite(a).all() and np.isfinite(e).all()
    P, V = 71, 42
    # right after a reset the simulated character is the clip pose: joint rotations (norm / tangent or angle) agree with the expert sample,
    # and so does the previous frame (InitHist samples the clip one query period earlier)
    np.testing.assert_allclose(a[7:7 + 52], e[7:7 + 52], atol=2e-6)
    np.testing.assert_allclose(a[P + 7:P + 7 + 52], e[P + 7:P + 7 + 52], atol=2e-6)
    # joint velocities: sim == clip after reset
    np.testing.assert_allclose(a[2 * P + 6:2 * P + V], e[2 * P + 6:2 * P + V], atol=2e-5)
    # normal / tangent pairs are orthonormal
    types = [j["Type"] for j in json.load(open(os.path.join(asset_root, "data/characters/humanoid3d.txt")))["Skeleton"]["Joints"]]
    k = 1
    for blk in [(1, "spherical")] + list(enumerate(types))[1:]:      # root rotation block, then the joints in file order
        if blk[1] == "spherical":
            n, t = a[k:k + 3], a[k + 3:k + 6]
            assert abs(np.dot(n, n) - 1) < 1e-6 and abs(np.dot(t, t) - 1) < 1e-6 and abs(np.dot(n, t)) < 1e-6
            k += 6
        elif blk[1] == "revolute":
            k += 1
    assert k == 7 + 52
    # root height above the ground = pose y
    pose, _ = o.get_pose()
    assert a[0] == pytest.approx(pose[1], abs=1e-12)
    # heading-local variant: the current root tangent has no z component (heading removed), end effectors are in the heading frame either way
    ol = Oracle(["--enable_amp_obs_local_root", "true"] + SPINKICK, asset_root)
    ol.reset(t0, 1.0, 20.0)
    al = ol.record_amp_obs_agent()
    assert abs(al[6]) < 1e-9
    np.testing.assert_allclose(al[7:7 + 52], a[7:7 + 52], atol=2e-6)   # joint part independent of the flag
    # after an action is applied the history is the pose the action was chosen from
    o.set_action(np.zeros(o.action_size))
    before = o.record_amp_obs_agent()[0:P]
    o.update(1.0 / 600.0)
    after = o.record_amp_obs_agent()
    # prev pose: joint rotations are heading independent -> equal to the "now" block before the update; root height too
    np.testing.assert_allclose(after[P + 7:P + 7 + 52], before[7:7 + 52], atol=1e-12)
    assert after[P] == pytest.approx(before[0], abs=1e-12)


# ---- behavioural pin against the REAL reference (SURVEY 8c): policies trained by the reference in Bullet 2.88 must work in this restatement
def _run_policy_in_oracle(o, actor, t0, steps=600):
    hidden = actor["hidden"]
    rew = []
    o.reset(t0, 0.0, 20.0)
    for _ in range(steps):
        if o.is_episode_end():
            break
        x = (o.record_state() - actor["s_norm_mean"]) / actor["s_norm_std"]
        for w, b in hidden:
            x = np.maximum(x @ w + b, 0.0)
        o.set_action((x @ actor["mean"][0] + actor["mean"][1]) * actor["a_norm_std"] + actor["a_norm_mean"])   # mode of the Gaussian actor
        for _ in range(20):
            o.update(1.0 / 600.0)
            if o.is_episode_end():
                break
        rew.append(o.calc_reward())
    return len(rew), float(np.mean(rew)), o.has_fallen(), o.get_time()


def _fixture_path(char, clip):
    return os.path.join(os.path.dirname(__file__), "golden", "policy_%s_%s_fp16.npz" % (char, clip))


def _fixture_actor(char="humanoid3d", clip="spinkick"):
    f = np.load(_fixture_path(char, clip))
    g = lambda k: f[k].astype(np.float64)
    return dict(hidden=[(g("w0"), g("b0")), (g("w1"), g("b1"))], mean=(g("wm"), g("bm")), s_norm_mean=g("s_mean"), s_norm_std=g("s_std"),
                a_norm_mean=g("a_mean"), a_norm_std=g("a_std"))


def test_pretrained_reference_policy_tracks_the_clip_in_the_oracle(asset_root):
    """The reference's own pretrained spin-kick policy (tests/golden fixture made from R/data/policies/humanoid3d/humanoid3d_spinkick.ckpt)
    drives the oracle for the whole 20 s test episode without falling and keeps the imitation reward high (0.90 measured).  The policy was
    trained in the real Bullet simulation, so this is a statistical pin of the restated physics + reward + observation against the reference."""
    o = Oracle(SPINKICK, asset_root)
    o.L.dmo_set_mode(o.h, 1)
    for t0 in (0.0, 0.5):
        n, mean_r, fallen, t = _run_policy_in_oracle(o, _fixture_actor(), t0)
        assert n == 600 and not fallen and t >= 20.0 - 1e-6, (t0, n, fallen, t)
        assert mean_r > 0.85, (t0, mean_r)


@pytest.mark.parametrize("char,clip,min_reward", [("humanoid3d", "walk", 0.8), ("humanoid3d", "backflip", 0.75), ("humanoid3d", "cartwheel", 0.8),
                                                   ("humanoid3d", "jump", 0.85), ("dog3d", "trot", 0.85), ("dog3d", "pace", 0.8), ("dog3d", "canter", 0.8),
                                                   ("dog3d", "spin", 0.75)])   # spin: --sync_char_root_rot true (0.44 when the sync only touched the pose, 0.80 with RotateOrigin)
def test_more_pretrained_policies_from_the_reference_tree(asset_root, char, clip, min_reward):
    """Same check for other skills: the committed fp16 fixture of the skill's policy on the committed assets where there is one (dog3d trot),
    else the TF1 checkpoint read directly (deepmimic_b200/tf_checkpoint.py) from a reference checkout."""
    if os.path.exists(_fixture_path(char, clip)):
        a, root = _fixture_actor(char, clip), asset_root
    else:
        root = reference_root()
        ckpt = os.path.join(root or "", "data/policies/%s/%s_%s.ckpt" % (char, char, clip))
        if not root or not os.path.exists(ckpt + ".index"):
            pytest.skip("reference checkout with pretrained policies not available (set DEEPMIMIC_REFERENCE_ROOT)")
        from deepmimic_b200.tf_checkpoint import load_actor
        a = load_actor(ckpt)
        a = {k: ([(w.astype(np.float64), b.astype(np.float64)) for w, b in v] if k == "hidden" else (tuple(x.astype(np.float64) for x in v) if k == "mean" else v.astype(np.float64)))
             for k, v in a.items()}
    o = Oracle(["--arg_file", "args/run_%s_%s_args.txt" % (char, clip)], root)
    o.L.dmo_set_mode(o.h, 1)
    n, mean_r, fallen, t = _run_policy_in_oracle(o, a, 0.0)
    assert n == 600 and not fallen, (clip, n, fallen)
    assert mean_r > min_reward, (clip, mean_r)


@pytest.mark.parametrize("arg_file,ckpt", [("args/run_amp_dog3d_trot_args.txt", "dog3d_amp/dog3d_amp_trot"), ("args/run_amp_humanoid3d_backflip_args.txt", "humanoid3d_amp/humanoid3d_amp_backflip"),
                                           ("args/run_amp_humanoid3d_crawl_args.txt", "humanoid3d_amp/humanoid3d_amp_crawl")])
def test_pretrained_amp_policies_stay_up_in_the_oracle(arg_file, ckpt):
    """The reference's AMP policies (scene imitate_amp: no phase input, state 226 / 346) are not phase-locked to the clip, so the imitation
    reward says little -- but they must keep the character going (back-flipping, crawling, trotting) for the whole 20 s without a fall."""
    ref = reference_root()
    path = os.path.join(ref or "", "data/policies", ckpt + ".ckpt")
    if not ref or not os.path.exists(path + ".index"):
        pytest.skip("reference checkout with pretrained policies not available (set DEEPMIMIC_REFERENCE_ROOT)")
    from deepmimic_b200.tf_checkpoint import load_actor
    a = load_actor(path)
    a = {k: ([(w.astype(np.float64), b.astype(np.float64)) for w, b in v] if k == "hidden" else (tuple(x.astype(np.float64) for x in v) if k == "mean" else v.astype(np.float64)))
         for k, v in a.items()}
    o = Oracle(["--arg_file", arg_file], ref)
    o.L.dmo_set_mode(o.h, 1)
    assert o.state_size == a["s_norm_mean"].shape[0]
    n, mean_r, fallen, t = _run_policy_in_oracle(o, a, 0.0)
    assert n == 600 and not fallen and t >= 20.0 - 1e-6, (arg_file, n, fallen, t)
