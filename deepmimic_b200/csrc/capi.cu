// C-ABI implementation (include/deepmimic_b200.h): host-side scene construction from the reference's asset
// formats, device model blob, launches of the sm_100a kernels.  No CPU fallback: every compute entry point
// launches CUDA work and fails loudly if the device / kernels are unavailable.
#include <cuda_runtime.h>

#include <algorithm>
#include <map>
#include <mutex>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <numeric>
#include <cstring>
#include <ctime>
#include <utility>
#include <memory>
#include <string>
#include <type_traits>
#include <vector>

#include "../../include/deepmimic_b200.h"
#include "host/assets.hpp"
#include "kernels/dm_model.cuh"

namespace dmk {
template <int W, int BLOCK, bool CLIPS>
__global__ void dm_observe_kernel(const DevModel*, DevState, const double*, const float*, const float*, ObsFan, int);
template <int W, int BLOCK, bool TASKV>
__global__ void dm_reset_kernel(const DevModel*, DevState, const double*, const float*, const float*, int, const double*, const double*, const double*,
                                unsigned long long, unsigned long long, int, const int*);
__global__ void dm_set_action_kernel(const DevModel*, DevState, const float*, int);
template <int W, int BLOCK, bool TASKV>
__global__ void dm_amp_obs_kernel(const DevModel*, DevState, const double*, const float*, const float*, float*, int, const double*, int, const int*);
template <int W, bool DEBUG, int VAR>
__global__ void dm_step_kernel(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
__global__ void dm_task_reset_kernel(const DevModel*, DevState, int);
__global__ void dm_task_observe_kernel(const DevModel*, DevState, float*, float*, int);
int dm_step_layout(int nl, int n, int chain_len, int maxrows, int W, StepLayout* L);
int dm_step_smem_bytes(const StepLayout& L, int tiles);

__global__ void dm_flags_kernel(DevState st, int32_t* out, int num_real_envs) {
    int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= num_real_envs) return;
    const int* f = st.flags + static_cast<size_t>(e) * kFlagInts;
    out[e * 4 + 0] = f[kFNeedAction]; out[e * 4 + 1] = f[kFDone]; out[e * 4 + 2] = f[kFTerminate]; out[e * 4 + 3] = f[kFValid];
}

// ---- multi-GPU exchange flags (dm_exchange_*): every rank owns one block {epoch[8], ack[8], status} that its peers write through P2P.
// epoch[r] = s + 1: rank r's rows of policy step s have arrived here; ack[r] = s + 1: rank r has finished reading the rows of step s there.
struct XchgFlags { unsigned long long epoch[8]; unsigned long long ack[8]; unsigned int status; unsigned int pad[31]; };
struct XchgPeers { int n; XchgFlags* f[8]; };
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// lane r publishes `value` into slot `me` of peer r's epoch (which = 0) or ack (which = 1) array.  The rows were stored by the preceding
// kernel of this stream; the system-scope fence + release store order them before the flag for the remote acquire load.
__global__ void dm_xchg_signal_kernel(XchgPeers P, int me, int which, unsigned long long value) {
    const int r = threadIdx.x;
    if (r >= P.n) return;
    __threadfence_system();
    st_release_sys(which == 0 ? &P.f[r]->epoch[me] : &P.f[r]->ack[me], value);
}
// lane r spins until this rank's own epoch[r] (which = 0) / ack[r] (which = 1) reaches `value`; gives up after `timeout_ns` and raises status
__global__ void dm_xchg_wait_kernel(XchgFlags* mine, int n, int which, unsigned long long value, unsigned long long timeout_ns) {
    const int r = threadIdx.x;
    if (r >= n) return;
    const unsigned long long* p = which == 0 ? &mine->epoch[r] : &mine->ack[r];
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while (ld_acquire_sys(p) < value) {
        unsigned long long t1;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
        if (t1 - t0 > timeout_ns) { atomicOr(&mine->status, 1u << which); return; }
        __nanosleep(200);
    }
}
}  // namespace dmk

static thread_local std::string g_err;
// every compute entry point: refuse host-only handles (dm_load_host) loudly, then select the handle's device
#define DM_DEVICE(h)                                                                                                             \
    do {                                                                                                                         \
        if ((h)->stream == nullptr) { g_err = "host-only handle (dm_load_host): no device state, and there is no CPU fallback"; return fail(); } \
        DM_CUDA(cudaSetDevice((h)->device));                                                                                     \
    } while (0)
#define DM_CUDA(call)                                                                                         \
    do {                                                                                                      \
        cudaError_t e_ = (call);                                                                              \
        if (e_ != cudaSuccess) { g_err = std::string(#call) + ": " + cudaGetErrorString(e_); return fail(); } \
    } while (0)

struct dm_handle {
    dmh::SceneAssets sa;
    dmk::DevModel hm;        // host copy of the model blob
    char *d_arena = nullptr, *p_arena = nullptr;   // the one device / pinned host allocation every fixed-size buffer below is carved from (carve_buffers)
    dmk::DevModel* d_model = nullptr;
    dmk::DevState st{};
    double* d_frame_times = nullptr;
    float* d_frames = nullptr;
    float* d_frame_vel = nullptr;
    double* d_inj[3] = {nullptr, nullptr, nullptr};
    int32_t* d_flags4 = nullptr;
    float *d_amp = nullptr, *p_amp = nullptr;                              // staging for dm_amp_obs_host
    float *d_goal = nullptr, *p_goal = nullptr;                            // staging for dm_goal_host (task scenes)
    dmk::ClipTable ctab{};                                                  // host copy of the clip dataset table (task scenes)
    dmk::ClipTable* d_ctab = nullptr; int* d_clip_inj = nullptr;           // device table; injected clip ids (reset / expert observations)
    int total_frames = 0;
    float *d_act = nullptr, *d_obs = nullptr, *d_rew = nullptr;            // staging for dm_step_host
    float *p_act = nullptr, *p_obs = nullptr, *p_rew = nullptr; int32_t* p_flags = nullptr;  // pinned host staging
    cudaStream_t stream = nullptr;
    int device = 0, num_envs = 0, padded_envs = 0, W = 32, tiles = 2, maxrows = 36, smem_bytes = 0;
    dmk::StepLayout lay{};
    uint64_t seed = 0, env_offset = 0;
    int64_t launches = 0;
    uint64_t amp_calls = 0;
    std::vector<double> st_off, st_scale, act_off, act_scale, act_min, act_max, st_groups;
    // dm_step_host: page-locked-ness of the caller's buffers, looked up once per pointer (cudaPointerGetAttributes is a driver call)
    std::vector<std::pair<const void*, bool>> pin_cache;
    // dm_step_host_timing: phase events of the last dm_step_host call (created by dm_set_timing)
    // dm_exchange_*: one allocation {XchgFlags | 2 x [obs world*N*S | rew world*N | done world*N]}, mapped into the peers through CUDA IPC
    int x_rank = 0, x_world = 0;
    char* x_base = nullptr;                       // this rank's allocation
    char* x_peer[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};   // every rank's allocation as seen from here ([x_rank] = x_base)
    size_t x_data_off = 0, x_parity_bytes = 0;
    bool timing = false;
    cudaEvent_t tev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    double host_ms[3] = {0, 0, 0};   // enqueue, wait (stream synchronize), staging copies
};

namespace {

int fail() { std::fprintf(stderr, "[deepmimic_b200] %s\n", g_err.c_str()); return 1; }

using dmh::Quat; using dmh::V3;
inline void put3(float* o, const V3& v, double s = 1.0) { o[0] = static_cast<float>(s * v.x); o[1] = static_cast<float>(s * v.y); o[2] = static_cast<float>(s * v.z); }
inline void putq(float* o, const Quat& q) { o[0] = static_cast<float>(q.x); o[1] = static_cast<float>(q.y); o[2] = static_cast<float>(q.z); o[3] = static_cast<float>(q.w); }

// Frame velocities of the clip, like cMotion::BuildFrameVel with cKinCharacter::CalcFrameVel -> cKinTree::CalcVel
// (R/DeepMimicCore/anim/Motion.cpp:170-191, anim/KinTree.cpp:1281-1316): world-frame rotation vector for the root,
// joint-local rotation vector for spherical joints, finite differences elsewhere.
std::vector<double> build_frame_vel(const dmh::CharModel& cm, const dmh::MotionClip& mc) {
    const int D = cm.pose_dim;
    std::vector<double> fv(static_cast<size_t>(mc.num_frames) * D, 0.0);
    for (int f = 0; f + 1 < mc.num_frames; ++f) {
        const double* a = mc.frame(f); const double* b = mc.frame(f + 1);
        const double dt = mc.frame_times[f + 1] - mc.frame_times[f];
        double* o = &fv[static_cast<size_t>(f) * D];
        for (int k = 0; k < 3; ++k) o[k] = (b[k] - a[k]) / dt;
        Quat q0(a[3], a[4], a[5], a[6]), q1(b[3], b[4], b[5], b[6]);
        V3 w = dmh::quat_to_rotvec(q1 * dmh::conj(q0));
        o[3] = w.x / dt; o[4] = w.y / dt; o[5] = w.z / dt; o[6] = 0;
        for (int j = 1; j < cm.num_joints(); ++j) {
            const auto& jd = cm.joints[j];
            const int p = jd.param_offset;
            if (jd.type == dmh::kSpherical) {
                Quat r0(a[p], a[p + 1], a[p + 2], a[p + 3]), r1(b[p], b[p + 1], b[p + 2], b[p + 3]);
                V3 wl = dmh::quat_to_rotvec(dmh::conj(r0) * r1);
                o[p] = wl.x / dt; o[p + 1] = wl.y / dt; o[p + 2] = wl.z / dt; o[p + 3] = 0;
            } else for (int k = 0; k < jd.param_size; ++k) o[p + k] = (b[p + k] - a[p + k]) / dt;
        }
    }
    if (mc.num_frames > 1) std::copy(fv.begin() + static_cast<size_t>(mc.num_frames - 2) * D, fv.begin() + static_cast<size_t>(mc.num_frames - 1) * D,
                                     fv.begin() + static_cast<size_t>(mc.num_frames - 1) * D);
    return fv;
}

// Digest the assets into the flat device model.  Frames follow cSimCharacter::BuildMultiBody
// (R/DeepMimicCore/sim/SimCharacter.cpp:789-946): every link frame sits at the body's COM with the body's orientation.
bool build_device_model(dm_handle& H) {
    const dmh::SceneAssets& sa = H.sa;
    const dmh::CharModel& cm = sa.character;
    dmk::DevModel& M = H.hm;
    std::memset(&M, 0, sizeof(M));
    const int nl = cm.num_joints();
    if (nl > dmk::kMaxLinks) { g_err = "character has more links than lanes (32)"; return false; }
    if (cm.joints[0].type != dmh::kNone) { g_err = "only floating-base characters (root joint type 'none') are supported"; return false; }
    const double sc = sa.cfg.world_scale;
    M.nl = nl; M.scale = static_cast<float>(sc);
    M.gravity[0] = static_cast<float>(sa.cfg.gravity.x * sc); M.gravity[1] = static_cast<float>(sa.cfg.gravity.y * sc); M.gravity[2] = static_cast<float>(sa.cfg.gravity.z * sc);
    M.friction = static_cast<float>(0.9 * 0.9);   // link 0.9 (sim/SimCharacter.cpp:26) x ground 0.9 (sim/Ground.cpp:17), Bullet multiplies them
    M.pose_dim = cm.pose_dim;
    M.phase_input = sa.ctrl.enable_phase_input; M.rec_world_root_pos = sa.ctrl.record_world_root_pos; M.rec_world_root_rot = sa.ctrl.record_world_root_rot;
    M.state_size = (M.phase_input ? 1 : 0) + 1 + nl * 9 + nl * 6;
    M.amp_local_root = sa.cfg.enable_amp_obs_local_root ? 1 : 0;
    {   // cSceneImitateAMP::GetAMPObsSize (SceneImitateAMP.cpp:75-84,214-258)
        int pose_sz = 1 + 6, nee = 0;
        for (int j = 0; j < nl; ++j) { const auto& jd = cm.joints[j]; if (jd.is_end_eff) ++nee; if (j > 0) pose_sz += (jd.type == dmh::kSpherical) ? 6 : jd.param_size; }
        M.amp_obs_size = 2 * (pose_sz + 3 * nee + 6 + (cm.pose_dim - cm.joints[0].param_size));
    }
    M.num_frames = sa.motion.num_frames; M.loop_motion = sa.motion.loop;
    M.end_at_clip_end = (!sa.motion.loop && sa.cfg.scene == "imitate") ? 1 : 0;   // cSceneImitateAMP::CheckTerminate skips the motion-over test (SceneImitateAMP.cpp:185-189)
    M.enable_fall_end = sa.cfg.enable_fall_end; M.enable_contact_fall = sa.cfg.enable_char_contact_fall; M.sync_root_pos = sa.cfg.sync_char_root_pos;
    M.sync_root_rot = sa.cfg.sync_char_root_rot; M.rand_rot_reset = sa.cfg.enable_rand_rot_reset;
    M.motion_dur = sa.motion.duration(); M.cycle_period = sa.motion.duration(); M.query_dt = 1.0 / sa.ctrl.query_rate;
    M.time_lim_min = sa.cfg.time_lim_min; M.time_lim_max = sa.cfg.time_lim_max; M.time_end_lim_max = sa.cfg.time_end_lim_max;
    M.total_mass = static_cast<float>(cm.total_mass());
    {   // AMP task scenes (dm_task.cuh)
        const dmh::SceneConfig& c = sa.cfg;
        M.task_kind = c.scene == "target_amp" ? dmk::kTaskTarget : c.scene == "heading_amp" ? dmk::kTaskHeading :
                      c.scene == "heading_amp_getup" ? dmk::kTaskHeadingGetup : c.scene == "strike_amp" ? dmk::kTaskStrike : dmk::kTaskNone;
        {   // heading_amp_getup / strike_amp (dm_task_ext.cuh)
            dmk::TaskExtParams& X = M.taskx;
            X.getup_time = 0.0;
            for (int id : c.getup_motion_ids) {
                if (id < 0 || id >= static_cast<int>(sa.clips.size())) { g_err = "--getup_motion_ids out of range"; return false; }
                X.getup_time = std::max(X.getup_time, sa.clips[id].duration());   // cSceneHeadingAMPGetup::CalcGetupTime (:262-287)
            }
            X.getup_height_root = c.getup_height_root; X.getup_height_head = c.getup_height_head; X.recover_episode_prob = c.recover_episode_prob;
            for (int k = 0; k < 3; ++k) { X.target_min[k] = c.target_min[k]; X.target_max[k] = c.target_max[k]; }
            X.target_radius = c.target_radius; X.hit_reset_time = c.target_hit_reset_time; X.tar_reward_scale = c.tar_reward_scale; X.hit_tar_speed = c.hit_tar_speed;
            X.init_hit_prob = c.init_hit_prob; X.tar_far_prob = c.tar_far_prob; X.tar_near_dist = c.tar_near_dist;
            X.head_id = c.head_id;
            if (X.head_id < 0 || X.head_id >= nl) { g_err = "--head_id out of range"; return false; }
            if (static_cast<int>(c.strike_bodies.size()) > dmk::kMaxTaskBodies || static_cast<int>(c.fail_tar_contact_bodies.size()) > dmk::kMaxTaskBodies) {
                g_err = "more than 4 --strike_bodies / --fail_tar_contact_bodies"; return false;
            }
            X.n_strike = static_cast<int>(c.strike_bodies.size()); X.n_fail = static_cast<int>(c.fail_tar_contact_bodies.size());
            for (int k = 0; k < dmk::kMaxTaskBodies; ++k) {
                X.strike_bodies[k] = k < X.n_strike ? c.strike_bodies[k] : 0; X.fail_bodies[k] = k < X.n_fail ? c.fail_tar_contact_bodies[k] : 0;
                if (X.strike_bodies[k] < 0 || X.strike_bodies[k] >= nl || X.fail_bodies[k] < 0 || X.fail_bodies[k] >= nl) { g_err = "strike / fail body id out of range"; return false; }
            }
            if (M.task_kind == dmk::kTaskStrike && X.n_strike == 0) { g_err = "strike_amp needs --strike_bodies"; return false; }
            if (M.task_kind == dmk::kTaskHeadingGetup && !(X.getup_time > 0.0)) { g_err = "heading_amp_getup needs --getup_motion_ids"; return false; }
        }
        dmk::TaskParams& T = M.task;
        T.timer_min = c.rand_target_time_min; T.timer_max = c.rand_target_time_max;
        T.max_target_dist = c.max_target_dist; T.target_succ_dist = c.target_succ_dist; T.tar_fail_dist = c.tar_fail_dist; T.pos_reward_scale = c.pos_reward_scale;
        T.max_heading_turn_rate = c.max_heading_turn_rate; T.sharp_turn_prob = c.sharp_turn_prob; T.speed_change_prob = c.speed_change_prob;
        T.tar_speed_min = c.tar_speed_min; T.tar_speed_max = c.tar_speed_max; T.vel_reward_scale = c.vel_reward_scale; T.tar_speed = c.tar_speed;
        T.enable_min_tar_vel = c.enable_min_tar_vel ? 1 : 0;
        M.task_seed = H.seed ^ 0x7461736b73ull;   // "tasks": a stream of its own next to the reset draws
        M.env_id_base = H.env_offset;
    }
    {
        const double* fb = sa.motion.frame(0); const double* fe = sa.motion.frame(sa.motion.num_frames - 1);
        M.cycle_delta[0] = static_cast<float>(fe[0] - fb[0]); M.cycle_delta[1] = 0.f; M.cycle_delta[2] = static_cast<float>(fe[2] - fb[2]);
    }
    double wsum = 0;
    for (const auto& j : cm.joints) wsum += std::fabs(j.diff_weight);
    int dof = 6, act_off = 0, maxlevel = 0, maxdepth = 5;
    std::vector<int> last_depth(nl, 5);
    for (int j = 0; j < nl; ++j) {
        const auto& jd = cm.joints[j]; const auto& bd = cm.bodies[j];
        dmk::DevLink& L = M.link[j];
        L.parent = jd.parent;
        const bool root = jd.parent < 0;
        if (root || jd.type == dmh::kFixed) { L.jtype = dmk::kJFixed; L.ndof = 0; }
        else if (jd.type == dmh::kRevolute) { L.jtype = dmk::kJRevolute; L.ndof = 1; }
        else if (jd.type == dmh::kSpherical) { L.jtype = dmk::kJSpherical; L.ndof = 3; }
        else { g_err = "unsupported joint type in character (planar / prismatic joints are outside the hot path)"; return false; }
        L.dof0 = dof; dof += L.ndof;
        L.level = root ? 0 : M.link[jd.parent].level + 1;
        maxlevel = std::max(maxlevel, L.level);
        L.nchild = 0;
        if (!root) {
            dmk::DevLink& P = M.link[jd.parent];
            if (P.nchild >= dmk::kMaxChildren) { g_err = "a link has more than 4 children"; return false; }
            P.child[P.nchild++] = j;
        }
        const int pd = root ? 5 : last_depth[jd.parent];
        L.depth0 = pd + 1;
        last_depth[j] = pd + L.ndof;
        L.last_depth = last_depth[j];
        maxdepth = std::max(maxdepth, last_depth[j]);
        if (last_depth[j] >= dmk::kMaxChain) { g_err = "dof chain too long"; return false; }
        if (root) for (int d = 0; d < 6; ++d) { M.chain_dof[j][d] = static_cast<uint8_t>(d); M.dof_depth[d] = static_cast<uint8_t>(d); M.dof_link[d] = 0; }
        else for (int d = 0; d <= pd; ++d) M.chain_dof[j][d] = M.chain_dof[jd.parent][d];
        for (int d = 0; d < L.ndof; ++d) { M.chain_dof[j][L.depth0 + d] = static_cast<uint8_t>(L.dof0 + d); M.dof_depth[L.dof0 + d] = static_cast<uint8_t>(L.depth0 + d); M.dof_link[L.dof0 + d] = static_cast<uint8_t>(j); }
        L.anc_mask = (root ? 0u : M.link[jd.parent].anc_mask) | (1u << j);
        // ---- frames
        Quat this_to_parent = dmh::euler_to_quat(jd.attach_theta), body_to_this = dmh::euler_to_quat(bd.attach_theta);
        Quat pb_to_parent; V3 pb_attach;
        if (!root) { pb_to_parent = dmh::euler_to_quat(cm.bodies[jd.parent].attach_theta); pb_attach = cm.bodies[jd.parent].attach_pt; }
        Quat parent_to_pb = dmh::conj(pb_to_parent);
        Quat body_to_pb = parent_to_pb * this_to_parent * body_to_this;
        putq(L.zrot, dmh::conj(body_to_pb));
        V3 e = dmh::rotate(parent_to_pb, jd.attach_pt) - dmh::rotate(parent_to_pb, pb_attach);
        V3 d = dmh::rotate(dmh::conj(body_to_this), bd.attach_pt);
        put3(L.evec, e, sc); put3(L.dvec, d, sc);
        put3(L.axis, dmh::rotate(dmh::conj(body_to_this), V3(0, 0, 1)));
        putq(L.child_rot, dmh::conj(body_to_this));
        put3(L.child_pos, -1.0 * dmh::rotate(dmh::conj(body_to_this), bd.attach_pt));
        put3(L.att_pt, jd.attach_pt); putq(L.att_rot, this_to_parent); put3(L.body_att, bd.attach_pt);
        // ---- mass properties at scaled size
        L.mass = static_cast<float>(bd.mass);
        const double m = bd.mass;
        if (bd.shape == dmh::kShapeBox) {
            L.shape = dmk::kSBox;
            const double hx = 0.5 * sc * bd.param[0], hy = 0.5 * sc * bd.param[1], hz = 0.5 * sc * bd.param[2];
            L.he[0] = static_cast<float>(hx); L.he[1] = static_cast<float>(hy); L.he[2] = static_cast<float>(hz);
            const double ix = m / 12.0 * (4 * hy * hy + 4 * hz * hz), iy = m / 12.0 * (4 * hx * hx + 4 * hz * hz), iz = m / 12.0 * (4 * hx * hx + 4 * hy * hy);
            L.inertiaB[0] = L.inertiaD[0] = static_cast<float>(ix); L.inertiaB[1] = L.inertiaD[1] = static_cast<float>(iy); L.inertiaB[2] = L.inertiaD[2] = static_cast<float>(iz);
            L.break_thr = static_cast<float>(0.02 * std::sqrt(hx * hx + hy * hy + hz * hz));
        } else if (bd.shape == dmh::kShapeCapsule) {
            L.shape = dmk::kSCapsule;
            const double r = 0.5 * sc * bd.param[0], hgt = sc * bd.param[1], hh = 0.5 * hgt;
            L.he[0] = static_cast<float>(r); L.he[1] = static_cast<float>(hh); L.he[2] = 0.f;
            // Bullet 2.88: inertia of the capsule's bounding box with CONVEX_DISTANCE_MARGIN (0.04, scaled units) added to every half extent
            // (btCapsuleShape::calculateLocalInertia)
            const double mg = 0.04, lx = 2 * (r + mg), ly = 2 * (r + hh + mg), lz = 2 * (r + mg), sm = m * 0.08333333;
            L.inertiaB[0] = static_cast<float>(sm * (ly * ly + lz * lz)); L.inertiaB[1] = static_cast<float>(sm * (lx * lx + lz * lz)); L.inertiaB[2] = static_cast<float>(sm * (lx * lx + ly * ly));
            // DeepMimic SPD model: exact capsule (cRBDUtil::BuildMomentInertiaCapsule, RBDUtil.cpp:667-694)
            const double c_vol = M_PI * r * r * hgt, hs_vol = M_PI * 2.0 / 3.0 * r * r * r, dens = m / (c_vol + 2 * hs_vol), cmass = c_vol * dens, hsm = hs_vol * dens;
            const double x = cmass * (0.25 * r * r + hgt * hgt / 12.0) + 2 * hsm * (0.4 * r * r + 0.375 * r * hgt + 0.25 * hgt * hgt), y = (0.5 * cmass + 0.8 * hsm) * r * r;
            L.inertiaD[0] = static_cast<float>(x); L.inertiaD[1] = static_cast<float>(y); L.inertiaD[2] = static_cast<float>(x);
            L.break_thr = static_cast<float>(0.02 * std::sqrt(2 * r * r + (r + hh) * (r + hh)));
        } else if (bd.shape == dmh::kShapeSphere) {
            L.shape = dmk::kSSphere;
            const double r = 0.5 * sc * bd.param[0];
            L.he[0] = static_cast<float>(r);
            const double i = 0.4 * m * r * r;
            for (int k = 0; k < 3; ++k) L.inertiaB[k] = L.inertiaD[k] = static_cast<float>(i);
            L.break_thr = static_cast<float>(0.02 * std::sqrt(3.0) * r);
        } else { g_err = "unsupported body shape (box / capsule / sphere only)"; return false; }
        L.fall_contact = bd.fall_contact; L.end_eff = jd.is_end_eff;
        L.kp = static_cast<float>(sc * sc * (root ? 0.0 : sa.ctrl.pd[j].kp)); L.kd = static_cast<float>(sc * sc * (root ? 0.0 : sa.ctrl.pd[j].kd));
        L.tlim = std::isfinite(jd.torque_lim) ? static_cast<float>(sc * sc * jd.torque_lim) : 3.0e38f;
        L.has_limit = (L.jtype == dmk::kJRevolute && jd.lim_low[0] <= jd.lim_high[1]) ? 1 : 0;   // sic: sim/SimCharacter.cpp:958
        L.lim_lo = static_cast<float>(jd.lim_low[0]); L.lim_hi = static_cast<float>(jd.lim_high[0]);
        L.joint_w = static_cast<float>(jd.diff_weight / wsum);
        L.pose_off = jd.param_offset; L.pose_size = jd.param_size;
        L.act_off = act_off; L.act_size = root ? 0 : (jd.type == dmh::kSpherical ? 3 : jd.param_size);
        act_off += L.act_size;
    }
    M.n = dof; M.maxlevel = maxlevel; M.action_size = act_off;
    M.cs = ((maxdepth + 1 + 7) / 8) * 8;
    if (M.n > dmk::kMaxDofs) { g_err = "too many dofs"; return false; }
    return true;
}

// static tables the agent reads once (cCtController / cCtCtrlUtil, SURVEY.md A.3, 8(c)(7))
void build_statics(dm_handle& H) {
    const auto& cm = H.sa.character; const auto& M = H.hm;
    H.st_off.assign(M.state_size, 0.0); H.st_scale.assign(M.state_size, 1.0); H.st_groups.assign(M.state_size, 0.0);
    if (M.phase_input) { H.st_off[0] = -0.5; H.st_scale[0] = 2.0; H.st_groups[0] = -1.0; }   // CtController.cpp:54-69,268-279,364-371
    H.act_off.assign(M.action_size, 0.0); H.act_scale.assign(M.action_size, 1.0); H.act_min.assign(M.action_size, 0.0); H.act_max.assign(M.action_size, 0.0);
    for (int j = 1; j < M.nl; ++j) {
        const auto& jd = cm.joints[j]; const auto& L = M.link[j];
        if (jd.type == dmh::kSpherical) {
            for (int k = 0; k < 3; ++k) { H.act_off[L.act_off + k] = 0; H.act_scale[L.act_off + k] = 2.0 / (2.0 * M_PI); H.act_min[L.act_off + k] = -2.0 * M_PI; H.act_max[L.act_off + k] = 2.0 * M_PI; }
        } else if (jd.type == dmh::kRevolute) {
            double lo = jd.lim_low[0], hi = jd.lim_high[0];
            if (!(hi >= lo)) { lo = -M_PI; hi = M_PI; }
            H.act_off[L.act_off] = -0.5 * (hi + lo); H.act_scale[L.act_off] = 0.5 / (hi - lo);
            const double mean = 0.5 * (hi + lo), delta = hi - lo;
            H.act_min[L.act_off] = mean - 2 * delta; H.act_max[L.act_off] = mean + 2 * delta;
        }
    }
}

// Calls f with std::integral_constant<int, 16> or <int, 32>, the handle's tile width, so that f can instantiate the kernels for it.
template <class F>
int with_width(const dm_handle* h, F&& f) { return h->W == 16 ? f(std::integral_constant<int, 16>{}) : f(std::integral_constant<int, 32>{}); }
// Calls f with std::true_type or std::false_type: the TASKV / CLIPS / DEBUG template flags of the kernels.
template <class F>
int with_flag(bool on, F&& f) { return on ? f(std::true_type{}) : f(std::false_type{}); }
// Epilogue of every launch: a bad launch configuration is reported here, and dm_get_counters counts the launch.
int launched(dm_handle* h) {
    DM_CUDA(cudaGetLastError());
    h->launches++;
    return 0;
}
bool is_task(const dm_handle* h) { return h->hm.task_kind != dmk::kTaskNone; }
constexpr int BLOCK = 64;   // threads per block of the per-environment kernels (reset, observations, AMP observations)

template <int W, bool DEBUG, int VAR>
int launch_step(dm_handle* h, double dt, int n_updates) {
    auto kern = dmk::dm_step_kernel<W, DEBUG, VAR>;
    // opt in to the large dynamic shared-memory carve-out; the limit is raised whenever a handle needs more than any earlier one on
    // this device (attributes are per device and per function: several handles of different sizes may live in one process)
    static std::mutex mu;
    static std::map<int, int> configured;   // device -> bytes configured for this instantiation
    {
        std::lock_guard<std::mutex> lock(mu);
        int& have = configured[h->device];
        if (h->smem_bytes > have) {
            DM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, h->smem_bytes));
            DM_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, 100));
            have = h->smem_bytes;
        }
    }
    const int grid = h->padded_envs / h->tiles;
    kern<<<grid, h->tiles * W, h->smem_bytes, h->stream>>>(h->d_model, h->st, h->d_frame_times, h->d_frames, dt, n_updates, h->sa.cfg.num_sim_substeps, h->lay);
    return launched(h);
}
template <int W, bool DEBUG>
int launch_update(dm_handle* h, double dt, int n_updates) {
    if (is_task(h)) {   // AMP task scenes: the instantiation that also advances the task block (no debug dumps there)
        if (DEBUG) { g_err = "dm_debug_enable is not available in the AMP task scenes"; return fail(); }
        if (h->hm.sync_root_rot) { g_err = "--sync_char_root_rot in an AMP task scene is not built"; return fail(); }
        return launch_step<W, false, dmk::kVarTask>(h, dt, n_updates);
    }
    if (h->hm.sync_root_rot) {   // --sync_char_root_rot true: the instantiation with the heading sync at clip wraps
        if (DEBUG) { g_err = "dm_debug_enable is not available with --sync_char_root_rot"; return fail(); }
        return launch_step<W, false, dmk::kVarRootRot>(h, dt, n_updates);
    }
    return launch_step<W, DEBUG, 0>(h, dt, n_updates);
}
// observation rows / imitation rewards into every destination of the fan; the task scenes read every environment's own active clip
int launch_observe_fan(dm_handle* h, const dmk::ObsFan& fan) {
    const size_t smem = static_cast<size_t>(BLOCK / h->W) * h->hm.state_size * sizeof(float);   // the block's observation rows, staged for 16-byte stores
    return with_width(h, [&](auto w) {
        return with_flag(is_task(h), [&](auto clips) {
            constexpr int W = decltype(w)::value;
            dmk::dm_observe_kernel<W, BLOCK, decltype(clips)::value><<<h->padded_envs / (BLOCK / W), BLOCK, smem, h->stream>>>(
                h->d_model, h->st, h->d_frame_times, h->d_frames, h->d_frame_vel, fan, h->num_envs);
            return launched(h);
        });
    });
}
int launch_observe(dm_handle* h, float* d_state, float* d_reward) {
    dmk::ObsFan fan{};
    fan.n = 1; fan.obs[0] = d_state; fan.rew[0] = d_reward; fan.done[0] = nullptr;
    return launch_observe_fan(h, fan);
}
// task scenes: per-environment clip of the dataset (`clip`: injected ids or nullptr), action history kept across resets
int launch_reset(dm_handle* h, int force, const double* kt, const double* mt, const double* th, const int* clip) {
    return with_width(h, [&](auto w) {
        return with_flag(is_task(h), [&](auto taskv) {
            constexpr int W = decltype(w)::value;
            dmk::dm_reset_kernel<W, BLOCK, decltype(taskv)::value><<<h->padded_envs / (BLOCK / W), BLOCK, 0, h->stream>>>(
                h->d_model, h->st, h->d_frame_times, h->d_frames, h->d_frame_vel, force, kt, mt, th, h->seed, h->env_offset, h->hm.test_mode, clip);
            return launched(h);
        });
    });
}
// AMP observations; `d_clips` (expert samples from per-environment dataset clips, task scenes) selects the CLIPS instantiation
int launch_amp(dm_handle* h, float* d_out, int expert, const double* d_times, const int* d_clips = nullptr) {
    return with_width(h, [&](auto w) {
        return with_flag(d_clips != nullptr, [&](auto clips) {
            constexpr int W = decltype(w)::value;
            dmk::dm_amp_obs_kernel<W, BLOCK, decltype(clips)::value><<<h->padded_envs / (BLOCK / W), BLOCK, 0, h->stream>>>(
                h->d_model, h->st, h->d_frame_times, h->d_frames, h->d_frame_vel, d_out, expert, d_times, h->num_envs, d_clips);
            return launched(h);
        });
    });
}
// Copies a field of the host model blob (h->hm) to the device blob, stream-ordered, and waits.  Host-only handles have no device blob.
int upload_model_field(dm_handle* h, const void* field, size_t bytes) {
    if (h->stream == nullptr) return 0;
    const size_t off = static_cast<size_t>(static_cast<const char*>(field) - reinterpret_cast<const char*>(&h->hm));
    DM_CUDA(cudaSetDevice(h->device));
    DM_CUDA(cudaMemcpyAsync(reinterpret_cast<char*>(h->d_model) + off, field, bytes, cudaMemcpyHostToDevice, h->stream));
    DM_CUDA(cudaStreamSynchronize(h->stream));
    return 0;
}
// The per-environment entry points take `env` from the caller: only real environments, never the padding ones dm_create froze.
bool bad_env(const dm_handle* h, int env, const char* fn) {
    if (env >= 0 && env < h->num_envs) return false;
    g_err = std::string(fn) + ": environment " + std::to_string(env) + " is out of range [0, " + std::to_string(h->num_envs) + ")";
    return true;
}

// A sub-allocator for the handle's fixed-size buffers: pieces aligned to 256 bytes, the alignment cudaMalloc gives.  Without a base it only
// adds up the size; with one it also sets the pointers.
struct Arena {
    char* base = nullptr;
    size_t bytes = 0;
    template <class T>
    void take(T*& p, size_t count) {
        bytes = (bytes + 255) / 256 * 256;
        p = base ? reinterpret_cast<T*>(base + bytes) : nullptr;
        bytes += count * sizeof(T);
    }
};
// every fixed-size buffer of a device handle, in one list for the sizing pass and the carving pass of dm_create
void carve_buffers(dm_handle& h, Arena& dev, Arena& pin) {
    const auto& M = h.hm;
    const size_t N = static_cast<size_t>(h.padded_envs), TF = static_cast<size_t>(h.total_frames), A = std::max(1, M.action_size);
    dev.take(h.d_model, 1);
    dev.take(h.st.sim, N * dmk::sim_stride(M.nl)); dev.take(h.st.time, N * dmk::kTimeDoubles); dev.take(h.st.flags, N * dmk::kFlagInts);
    dev.take(h.st.manifold, N * M.nl * dmk::kManifoldFloats); dev.take(h.st.hist, N * 2 * M.pose_dim);
    dev.take(h.d_frame_times, TF); dev.take(h.d_frames, TF * M.pose_dim); dev.take(h.d_frame_vel, TF * M.pose_dim);   // mocap tables
    dev.take(h.d_flags4, N * 4); dev.take(h.d_amp, N * M.amp_obs_size);
    dev.take(h.d_act, N * A); dev.take(h.d_obs, N * M.state_size); dev.take(h.d_rew, N);
    for (auto& p : h.d_inj) dev.take(p, N);
    pin.take(h.p_act, N * A); pin.take(h.p_obs, N * M.state_size); pin.take(h.p_rew, N); pin.take(h.p_flags, N * 4); pin.take(h.p_amp, N * M.amp_obs_size);
    if (is_task(&h)) {
        dev.take(h.st.task, N * dmk::kTaskDoubles); dev.take(h.st.taskx, N * dmk::kTaskExtDoubles); dev.take(h.st.clip, N);
        dev.take(h.d_clip_inj, N); dev.take(h.d_ctab, 1); dev.take(h.d_goal, N * 4);
        pin.take(h.p_goal, N * 4);
    }
}

}  // namespace

// Launch plan of dm_step_kernel: tile width, row capacity, shared-memory layout, environments per block (one block per SM: as many
// environments per block as shared memory and kStepMaxThreads allow, balanced over the SMs), padded environment count.  Pure host arithmetic
// (also reachable without a device through dm_plan_launch, for the CPU tests of the one-wave property).
static bool plan_launch(dm_handle& H, int num_envs, int smem_optin, int sms) {
    const auto& M = H.hm;
    H.W = (M.nl <= 16) ? 16 : 32;   // lanes per environment: one lane per link
    H.maxrows = dmk::dm_step_y_stride(H.W);   // humanoid3d: 8 foot points x 3 + limit rows <= 28 of 32; dog3d: 4 feet x 4 points x 3 + 4 limit rows = 52
    int chain_len = 0;
    for (int j = 0; j < M.nl; ++j) chain_len = std::max(chain_len, M.link[j].last_depth + 1);
    dmk::dm_step_layout(M.nl, M.n, chain_len, H.maxrows, H.W, &H.lay);
    const int per_env = H.lay.env_floats * 4;
    const int hot = H.lay.hot_floats * 4 + 1024;
    const int max_tiles = std::min(dmk::kStepMaxThreads / H.W, (smem_optin - hot) / per_env);
    const int min_tiles = (H.W == 16) ? 2 : 1;   // W = 16: two environments share a warp
    if (max_tiles < min_tiles) {
        g_err = "not enough shared memory per block for one environment tile (need " + std::to_string(hot + min_tiles * per_env) + " bytes, the device offers " +
                std::to_string(static_cast<long long>(smem_optin)) + ")";
        return false;
    }
    int tiles = std::min(max_tiles, std::max(min_tiles, (num_envs + sms - 1) / sms));
    if (H.W == 16 && (tiles & 1)) tiles = (tiles + 1 <= max_tiles) ? tiles + 1 : tiles - 1;   // whole warps; tiles >= 2 here, so tiles - 1 >= 2 when odd
    H.tiles = tiles;
    const int quantum = (tiles * (64 / H.W)) / std::__gcd(tiles, 64 / H.W);   // multiple of both the update block and the 64-thread policy blocks
    H.padded_envs = ((num_envs + quantum - 1) / quantum) * quantum;
    H.smem_bytes = dmk::dm_step_smem_bytes(H.lay, H.tiles) + 1024;
    return true;
}

extern "C" {

const char* dm_last_error(void) { return g_err.c_str(); }
void dm_set_last_error(const char* msg) { g_err = msg ? msg : ""; }   // other translation units of the library (mlp_capi.cu) report through the same string

// host half of dm_create: argument / asset loading and the flat model (no device work)
static bool load_host_model(dm_handle& H, const char* asset_root, int argc, const char** argv) {
    try {
        std::vector<std::string> args(argv, argv + argc);
        dmh::ArgParser ap;
        ap.LoadArgs(args);
        std::string root = asset_root ? asset_root : "", arg_file;
        if (ap.ParseString("arg_file", arg_file) && !ap.LoadFile(dmh::resolve_path(root, arg_file))) throw std::runtime_error("Failed to load args from: " + arg_file);
        std::string timer_type;
        if (ap.ParseString("timer_type", timer_type) && timer_type != "" && timer_type != "uniform")   // cTimer::ParseTypeStr (util/Timer.cpp:26-43)
            throw std::runtime_error("Unsupported timer type " + timer_type + " (supported: uniform)");
        H.sa = dmh::load_scene_assets(ap, root);
        // scenes on the accelerated path: "imitate" and its AMP variant (same character, controller, clip and dynamics; AMP observations on top).
        // The AMP task scenes (heading / target / dribble / strike) add goals, task rewards and clip datasets that are not built: refuse them loudly.
        // options of the reference's scene that the batched path does not implement are refused, never ignored
        {
            const dmh::SceneConfig& c = H.sa.cfg;
            std::vector<std::string> v;
            if (!c.char_ctrl.empty() && c.char_ctrl != "ct_pd") throw std::runtime_error("Unsupported character controller: " + c.char_ctrl + " (supported: ct_pd)");
            if (ap.ParseStrings("character_files", v) && v.size() > 1) throw std::runtime_error("Unsupported: more than one character per scene");
            if (ap.ParseStrings("char_types", v) && !v.empty() && v[0] != "general") throw std::runtime_error("Unsupported character type: " + v[0] + " (supported: general)");
            bool soft = false;
            if (ap.ParseBool("enable_char_soft_contact", soft) && soft) throw std::runtime_error("Unsupported: --enable_char_soft_contact true");
            if (c.enable_root_rot_fail) throw std::runtime_error("Unsupported: --enable_root_rot_fail true");
            if (!c.terrain_file.empty()) {   // cGroundBuilder: only the flat plane (data/terrain/plane.txt) is on the path
                dmh::Json t = dmh::Json::parseFile(dmh::resolve_path(root, c.terrain_file));
                if (t["Type"].asString("") != "plane") throw std::runtime_error("Unsupported terrain type: " + t["Type"].asString("") + " (supported: plane)");
            }
        }
        // Scenes on the accelerated path: imitate, imitate_amp, and the AMP task scenes target_amp / heading_amp (goals, task rewards, clip
        // datasets; validated on hardware against the oracle in round 2: tests/test_task_scenes_gpu.py).  heading_amp_getup / strike_amp have
        // their device code written and host-checked but are not validated on hardware: opt-in with DM_EXPERIMENTAL_TASK_SCENES=1.  Every other
        // scene name is refused.
        const char* exp_env = std::getenv("DM_EXPERIMENTAL_TASK_SCENES");
        const bool experimental = exp_env != nullptr && exp_env[0] == '1';
        const bool task_scene = H.sa.cfg.is_task_scene();   // target_amp, heading_amp, heading_amp_getup, strike_amp
        const std::string& scn = H.sa.cfg.scene;
        const bool validated = scn == "imitate" || scn == "imitate_amp" || scn == "target_amp" || scn == "heading_amp";
        if (!validated && !(task_scene && experimental))
            throw std::runtime_error("Unsupported scene: " + scn + " (supported: imitate, imitate_amp, target_amp, heading_amp)");
        if (H.sa.clips.size() != 1 && !task_scene)
            throw std::runtime_error("Unsupported kinematic controller: clips with more than one clip outside the AMP task scenes (supported: motion)");
        if (static_cast<int>(H.sa.clips.size()) > dmk::kMaxClips) throw std::runtime_error("clip dataset larger than the device clip table (" + std::to_string(dmk::kMaxClips) + ")");
    } catch (const std::exception& e) { g_err = e.what(); return false; }
    if (!build_device_model(H)) return false;
    build_statics(H);
    return true;
}

dm_handle* dm_load_host(const char* asset_root, int argc, const char** argv) {
    std::unique_ptr<dm_handle> h(new dm_handle());
    if (!load_host_model(*h, asset_root, argc, argv)) { fail(); return nullptr; }
    return h.release();
}

int dm_plan_launch(dm_handle* h, int num_envs, int smem_bytes_per_block, int num_sms, int* out) {
    if (!h || num_envs <= 0 || num_sms <= 0) { g_err = "dm_plan_launch: bad arguments"; return fail(); }
    dm_handle tmp;
    tmp.hm = h->hm;
    if (!plan_launch(tmp, num_envs, smem_bytes_per_block, num_sms)) return fail();
    out[0] = tmp.W; out[1] = tmp.tiles; out[2] = tmp.padded_envs / tmp.tiles; out[3] = tmp.smem_bytes; out[4] = tmp.maxrows; out[5] = tmp.lay.env_floats;
    out[6] = tmp.lay.hot_floats; out[7] = tmp.lay.oY; out[8] = tmp.padded_envs;
    return 0;
}

int dm_get_model_info(dm_handle* h, int kind, int* out) {
    const auto& M = h->hm;
    switch (kind) {
        case DM_INFO_PARENTS: for (int j = 0; j < M.nl; ++j) out[j] = M.link[j].parent; break;
        case DM_INFO_JOINT_TYPES: for (int j = 0; j < M.nl; ++j) out[j] = M.link[j].jtype; break;
        case DM_INFO_DOF_OFFSETS: for (int j = 0; j < M.nl; ++j) out[j] = M.link[j].dof0; break;
        case DM_INFO_POSE_OFFSETS: for (int j = 0; j < M.nl; ++j) out[j] = M.link[j].pose_off; break;
        case DM_INFO_FALL_BODIES: for (int j = 0; j < M.nl; ++j) out[j] = M.link[j].fall_contact; break;
        case DM_INFO_END_EFFECTORS: for (int j = 0; j < M.nl; ++j) out[j] = M.link[j].end_eff; break;
        case DM_INFO_LAYOUT: out[0] = M.nl; out[1] = M.n; out[2] = M.cs; out[3] = M.maxlevel; out[4] = M.num_frames; out[5] = M.loop_motion; break;
        default: g_err = "dm_get_model_info: bad kind"; return fail();
    }
    return 0;
}

// Per-link model constants as the kernels use them (24 doubles per link): mass, Bullet inertia[3], DeepMimic inertia[3], dvec[3], evec[3],
// zrot (x,y,z,w), axis[3], half extents[3], breaking threshold.  Scaled units.  For the independent known-answer tests of the loader.
int dm_get_link_table(dm_handle* h, double* out) {
    const auto& M = h->hm;
    for (int j = 0; j < M.nl; ++j) {
        const dmk::DevLink& L = M.link[j];
        double* o = out + 24 * j;
        o[0] = L.mass;
        for (int k = 0; k < 3; ++k) { o[1 + k] = L.inertiaB[k]; o[4 + k] = L.inertiaD[k]; o[7 + k] = L.dvec[k]; o[10 + k] = L.evec[k]; o[17 + k] = L.axis[k]; o[20 + k] = L.he[k]; }
        for (int k = 0; k < 4; ++k) o[13 + k] = L.zrot[k];
        o[23] = L.break_thr;
    }
    return 0;
}

dm_handle* dm_create(const char* asset_root, int argc, const char** argv, int num_envs, int device, uint64_t seed, uint64_t global_env_offset) {
    std::unique_ptr<dm_handle> h(new dm_handle());
    if (!load_host_model(*h, asset_root, argc, argv)) { fail(); return nullptr; }
    if (num_envs <= 0) { g_err = "num_envs must be positive"; fail(); return nullptr; }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) { g_err = "no CUDA device available: deepmimic_b200 has no CPU fallback"; fail(); return nullptr; }
    auto chk = [&](cudaError_t e, const char* what) { if (e != cudaSuccess) { g_err = std::string(what) + ": " + cudaGetErrorString(e); return false; } return true; };
    if (!chk(cudaSetDevice(device), "cudaSetDevice")) { fail(); return nullptr; }
    h->device = device; h->seed = seed; h->env_offset = global_env_offset; h->num_envs = num_envs;
    h->hm.task_seed = seed ^ 0x7461736b73ull; h->hm.env_id_base = global_env_offset;   // the model blob is uploaded below
    const auto& M = h->hm;
    {
        cudaDeviceProp prop;
        if (!chk(cudaGetDeviceProperties(&prop, device), "cudaGetDeviceProperties")) { fail(); return nullptr; }
        if (!plan_launch(*h, num_envs, static_cast<int>(prop.sharedMemPerBlockOptin), prop.multiProcessorCount)) { fail(); return nullptr; }
    }
    const size_t N = static_cast<size_t>(h->padded_envs);
    const int ss = dmk::sim_stride(M.nl);
    // mocap tables: the frames of every clip of the scene, concatenated (one clip unless --kin_ctrl clips; clip 0 = the model's clip)
    h->total_frames = 0;
    h->ctab = dmk::ClipTable{};
    h->ctab.num_clips = static_cast<int>(h->sa.clips.size());
    for (size_t c = 0; c < h->sa.clips.size(); ++c) {
        const dmh::MotionClip& mc = h->sa.clips[c];
        dmk::ClipInfo& ci = h->ctab.info[c];
        ci.dur = mc.duration(); ci.frame_off = h->total_frames; ci.num_frames = mc.num_frames; ci.loop = mc.loop ? 1 : 0;
        const double* fb = mc.frame(0); const double* fe = mc.frame(mc.num_frames - 1);
        ci.cycle_delta[0] = static_cast<float>(fe[0] - fb[0]); ci.cycle_delta[1] = 0.f; ci.cycle_delta[2] = static_cast<float>(fe[2] - fb[2]);
        h->ctab.cdf[c] = h->sa.clip_cdf[c];
        ci.is_getup = std::find(h->sa.cfg.getup_motion_ids.begin(), h->sa.cfg.getup_motion_ids.end(), static_cast<int>(c)) != h->sa.cfg.getup_motion_ids.end() ? 1 : 0;
        h->total_frames += mc.num_frames;
    }
    const size_t TF = static_cast<size_t>(h->total_frames);
    Arena dev, pin;
    carve_buffers(*h, dev, pin);   // sizing pass
    bool ok = chk(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking), "cudaStreamCreate") &&
              chk(cudaMalloc(&h->d_arena, dev.bytes), "cudaMalloc") && chk(cudaMallocHost(&h->p_arena, pin.bytes), "cudaMallocHost") &&
              chk(cudaMemset(h->d_arena, 0, dev.bytes), "cudaMemset");
    if (!ok) { fail(); dm_destroy(h.release()); return nullptr; }
    dev = Arena{h->d_arena}; pin = Arena{h->p_arena};
    carve_buffers(*h, dev, pin);   // carving pass
    h->st.num_envs = h->padded_envs; h->st.num_real = h->num_envs;
    h->st.ctab = h->d_ctab;
    std::vector<float> frames(TF * M.pose_dim), fvel(frames.size());
    std::vector<double> ftimes(TF);
    for (size_t c = 0; c < h->sa.clips.size(); ++c) {
        const dmh::MotionClip& mc = h->sa.clips[c];
        const std::vector<double> fv = build_frame_vel(h->sa.character, mc);
        const size_t off = static_cast<size_t>(h->ctab.info[c].frame_off);
        std::copy(mc.frame_times.begin(), mc.frame_times.end(), ftimes.begin() + off);
        for (size_t i = 0; i < mc.frames.size(); ++i) { frames[off * M.pose_dim + i] = static_cast<float>(mc.frames[i]); fvel[off * M.pose_dim + i] = static_cast<float>(fv[i]); }
    }
    ok = chk(cudaMemcpy(h->d_model, &h->hm, sizeof(dmk::DevModel), cudaMemcpyHostToDevice), "memcpy model") &&
         chk(cudaMemcpy(h->d_frame_times, ftimes.data(), sizeof(double) * TF, cudaMemcpyHostToDevice), "memcpy ft") &&
         chk(cudaMemcpy(h->d_frames, frames.data(), sizeof(float) * frames.size(), cudaMemcpyHostToDevice), "memcpy frames") &&
         chk(cudaMemcpy(h->d_frame_vel, fvel.data(), sizeof(float) * fvel.size(), cudaMemcpyHostToDevice), "memcpy fvel") &&
         (!is_task(h.get()) || chk(cudaMemcpy(h->d_ctab, &h->ctab, sizeof(dmk::ClipTable), cudaMemcpyHostToDevice), "memcpy clip table"));
    if (ok && h->padded_envs > h->num_envs) {
        // padding environments (the step kernel works on whole blocks): marked done once and for all, so that every kernel skips them.  Left
        // alive they would stand on both feet without ever receiving an action -- 26 constraint rows each, the slowest block of the launch
        // (found with tools/section_profile.py in round 2: the last block set the kernel time).
        std::vector<int> fl(static_cast<size_t>(h->padded_envs - h->num_envs) * dmk::kFlagInts, 0);
        for (int e = 0; e < h->padded_envs - h->num_envs; ++e) { fl[static_cast<size_t>(e) * dmk::kFlagInts + dmk::kFDone] = 1; fl[static_cast<size_t>(e) * dmk::kFlagInts + dmk::kFValid] = 1; }
        ok = chk(cudaMemcpy(h->st.flags + static_cast<size_t>(h->num_envs) * dmk::kFlagInts, fl.data(), fl.size() * sizeof(int), cudaMemcpyHostToDevice), "memcpy padding flags");
    }
    if (ok) {
        // initial PD targets: identity / TargetTheta0 (cPDController::Init, PDController.cpp:99-112)
        std::vector<float> sim(N * ss, 0.f);
        for (size_t e = 0; e < N; ++e) for (int j = 0; j < M.nl; ++j) {
            float* t = &sim[e * ss + 16 + 8 * M.nl + 4 * j];
            if (M.link[j].jtype == dmk::kJSpherical) { t[0] = t[1] = t[2] = 0.f; t[3] = 1.f; }
            else t[0] = static_cast<float>(h->sa.ctrl.pd[j].target_theta[0]);
        }
        ok = chk(cudaMemcpy(h->st.sim, sim.data(), sim.size() * sizeof(float), cudaMemcpyHostToDevice), "memcpy sim");
    }
    if (!ok) { fail(); dm_destroy(h.release()); return nullptr; }
    if (dm_reset(h.get(), 1, nullptr, nullptr, nullptr) != 0 || dm_sync(h.get()) != 0) { dm_destroy(h.release()); return nullptr; }
    return h.release();
}

int dm_exchange_destroy(dm_handle* h);
void dm_destroy(dm_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    dm_exchange_destroy(h);
    cudaFree(h->d_arena); cudaFreeHost(h->p_arena); cudaFree(h->st.pdbg);
    for (auto& e : h->tev) if (e) cudaEventDestroy(e);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

int dm_get_dims(dm_handle* h, dm_dims* o) {
    const auto& M = h->hm;
    o->num_envs = h->num_envs; o->num_joints = M.nl; o->pose_dim = M.pose_dim; o->num_dofs = M.n; o->state_size = M.state_size; o->goal_size = M.task_kind == dmk::kTaskNone ? 0 : (M.task_kind >= dmk::kTaskHeadingGetup ? 4 : 3); o->amp_obs_size = M.amp_obs_size;
    o->action_size = M.action_size; o->snapshot_size = 29 + 59 * M.nl;
    o->num_update_substeps = h->sa.cfg.num_update_substeps;
    o->updates_per_action = 20;
    o->motion_duration = M.motion_dur;
    return 0;
}
// cScene::GetName of the configured scene (SceneImitate.cpp:209, SceneImitateAMP.cpp:211, SceneTargetAMP.cpp:233, SceneHeadingAMP.cpp:153, ...)
int dm_get_scene_name(dm_handle* h, char* out, int cap) {
    const std::string& sc = h->sa.cfg.scene;
    const char* name = sc == "imitate_amp" ? "Imitate AMP" : sc == "target_amp" ? "Target AMP" : sc == "heading_amp" ? "Heading AMP" :
                       sc == "heading_amp_getup" ? "Heading AMP Getup" : sc == "strike_amp" ? "Strike AMP" : "Imitate";
    if (cap <= 0) { g_err = "dm_get_scene_name: empty buffer"; return fail(); }
    std::snprintf(out, static_cast<size_t>(cap), "%s", name);
    return 0;
}
int dm_get_static(dm_handle* h, int kind, double* out) {
    const std::vector<double>* v = nullptr;
    switch (kind) {
        case DM_STATE_OFFSET: v = &h->st_off; break; case DM_STATE_SCALE: v = &h->st_scale; break; case DM_ACTION_OFFSET: v = &h->act_off; break;
        case DM_ACTION_SCALE: v = &h->act_scale; break; case DM_ACTION_BOUND_MIN: v = &h->act_min; break; case DM_ACTION_BOUND_MAX: v = &h->act_max; break;
        case DM_STATE_NORM_GROUPS: v = &h->st_groups; break; default: g_err = "dm_get_static: bad kind"; return fail();
    }
    std::copy(v->begin(), v->end(), out);
    return 0;
}
void* dm_stream(dm_handle* h) { return h->stream; }
int dm_sync(dm_handle* h) { DM_DEVICE(h); DM_CUDA(cudaStreamSynchronize(h->stream)); return 0; }
int dm_set_mode(dm_handle* h, int mode) {
    h->hm.test_mode = mode;   // the reset kernel takes it as an argument; the task scenes also read it inside the kernels (test-mode get-ups, rewards)
    return is_task(h) ? upload_model_field(h, &h->hm.test_mode, sizeof(int)) : 0;
}
// the reset kernel reads the episode time limits from the model blob: both are uploaded as one field
static_assert(offsetof(dmk::DevModel, time_lim_max) == offsetof(dmk::DevModel, time_lim_min) + sizeof(double), "time limits must be adjacent");
// cRLSceneSimChar::SetSampleCount -> UpdateTimerParams (RLSceneSimChar.cpp:223-227,330-347): the episode time limits move from
// (time_lim_min, time_lim_max) to (time_end_lim_min, time_end_lim_max) with lerp = clamp(count / anneal_samples, 0, 1)^4.
int dm_set_sample_count(dm_handle* h, long long count) {
    const dmh::SceneConfig& c = h->sa.cfg;
    if (c.anneal_samples <= 0) return 0;
    double t = static_cast<double>(count) / static_cast<double>(c.anneal_samples);
    t = std::min(std::max(t, 0.0), 1.0);
    const double lerp = std::pow(t, 4.0);
    auto mix = [lerp](double a, double b) { return (a == b) ? a : (1.0 - lerp) * a + lerp * b; };   // cMathUtil::Lerp; a == b keeps infinities finite-safe
    h->hm.time_lim_min = mix(c.time_lim_min, c.time_end_lim_min);
    h->hm.time_lim_max = mix(c.time_lim_max, c.time_end_lim_max);
    return upload_model_field(h, &h->hm.time_lim_min, 2 * sizeof(double));
}
// Episode time limits set directly (both train-mode bounds): bench.py and tests that want a fixed limit without the annealing schedule.
int dm_set_time_limits(dm_handle* h, double tmin, double tmax) {
    if (!(tmin > 0.0) || !(tmax >= tmin)) { g_err = "dm_set_time_limits: need 0 < min <= max"; return fail(); }
    h->hm.time_lim_min = tmin; h->hm.time_lim_max = tmax;
    return upload_model_field(h, &h->hm.time_lim_min, 2 * sizeof(double));
}
int dm_get_time_limits(dm_handle* h, double* out) {
    out[0] = h->hm.time_lim_min; out[1] = h->hm.time_lim_max; out[2] = h->hm.time_end_lim_max;
    return 0;
}

int dm_reset_clips(dm_handle* h, int force_all, const int* h_clip, const double* kt, const double* mt, const double* th) {
    DM_DEVICE(h);
    const double* src[3] = {kt, mt, th}; const double* dev[3] = {nullptr, nullptr, nullptr};
    std::vector<double> tmp(h->padded_envs);
    for (int k = 0; k < 3; ++k) if (src[k]) {
        for (int e = 0; e < h->padded_envs; ++e) tmp[e] = src[k][e < h->num_envs ? e : h->num_envs - 1];
        DM_CUDA(cudaMemcpyAsync(h->d_inj[k], tmp.data(), sizeof(double) * h->padded_envs, cudaMemcpyHostToDevice, h->stream));
        DM_CUDA(cudaStreamSynchronize(h->stream));
        dev[k] = h->d_inj[k];
    }
    const int* dclip = nullptr;
    if (h_clip) {
        if (h->hm.task_kind == dmk::kTaskNone) { g_err = "dm_reset_clips: clip ids can only be injected in the AMP task scenes"; return fail(); }
        std::vector<int> ct(h->padded_envs);
        for (int e = 0; e < h->padded_envs; ++e) {
            ct[e] = h_clip[e < h->num_envs ? e : h->num_envs - 1];
            if (ct[e] < 0 || ct[e] >= h->ctab.num_clips) { g_err = "dm_reset_clips: clip id out of range"; return fail(); }
        }
        DM_CUDA(cudaMemcpyAsync(h->d_clip_inj, ct.data(), sizeof(int) * h->padded_envs, cudaMemcpyHostToDevice, h->stream));
        DM_CUDA(cudaStreamSynchronize(h->stream));
        dclip = h->d_clip_inj;
    }
    if (launch_reset(h, force_all, dev[0], dev[1], dev[2], dclip)) return 1;
    if (is_task(h)) {   // cSceneTargetAMP::Reset's own part for the environments that were just reset
        dmk::dm_task_reset_kernel<<<(h->padded_envs + 127) / 128, 128, 0, h->stream>>>(h->d_model, h->st, h->padded_envs);
        return launched(h);
    }
    return 0;
}
int dm_reset(dm_handle* h, int force_all, const double* kt, const double* mt, const double* th) { return dm_reset_clips(h, force_all, nullptr, kt, mt, th); }
int dm_get_clip_table(dm_handle* h, int* num_clips, double* h_dur, double* h_cdf) {
    const int n = static_cast<int>(h->sa.clips.size());
    if (num_clips) *num_clips = n;
    for (int c = 0; c < n; ++c) { if (h_dur) h_dur[c] = h->sa.clips[c].duration(); if (h_cdf) h_cdf[c] = h->sa.clip_cdf[c]; }
    return 0;
}
int dm_set_action(dm_handle* h, const float* d_actions) {
    DM_DEVICE(h);
    const int total = h->num_envs * h->hm.nl;
    dmk::dm_set_action_kernel<<<(total + 127) / 128, 128, 0, h->stream>>>(h->d_model, h->st, d_actions, h->num_envs);
    return launched(h);
}
int dm_update(dm_handle* h, double dt, int n_updates) {
    DM_DEVICE(h);
    bool dbg = h->st.pdbg != nullptr;
#ifdef DM_PROFILE
    dbg = false;   // profile build: the production kernel writes its per-warp section counters into the debug buffer
#endif
    return with_width(h, [&](auto w) { return with_flag(dbg, [&](auto debug) { return launch_update<decltype(w)::value, decltype(debug)::value>(h, dt, n_updates); }); });
}
static int launch_task_observe(dm_handle* h, float* d_goal, float* d_reward) {
    dmk::dm_task_observe_kernel<<<(h->num_envs + 127) / 128, 128, 0, h->stream>>>(h->d_model, h->st, d_goal, d_reward, h->num_envs);
    return launched(h);
}
int dm_observe(dm_handle* h, float* d_state, float* d_reward) {
    DM_DEVICE(h);
    const bool task = is_task(h);   // the task scenes replace CalcReward (SceneTargetAMP.cpp:3-80, SceneHeadingAMP.cpp:3-48)
    float* d_imitate_reward = task ? nullptr : d_reward;
    if ((d_state != nullptr || d_imitate_reward != nullptr) && launch_observe(h, d_state, d_imitate_reward)) return 1;
    if (task && d_reward != nullptr) return launch_task_observe(h, nullptr, d_reward);
    return 0;
}
int dm_record_state(dm_handle* h, float* d_out) { return dm_observe(h, d_out, nullptr); }
// cSceneImitate::CalcRewardImitate in every scene: in the AMP task scenes (where CalcReward is the task reward) against the environment's
// active clip of the dataset -- BASELINE.json config 5 records it beside the AMP observations.
int dm_calc_reward_imitate(dm_handle* h, float* d_out) {
    DM_DEVICE(h);
    return launch_observe(h, nullptr, d_out);
}
int dm_record_goal(dm_handle* h, float* d_out) {
    if (h->hm.task_kind == dmk::kTaskNone) return 0;
    DM_DEVICE(h);
    return launch_task_observe(h, d_out, nullptr);
}
int dm_goal_host(dm_handle* h, float* h_out) {
    if (h->hm.task_kind == dmk::kTaskNone) return 0;
    DM_DEVICE(h);
    if (launch_task_observe(h, h->d_goal, nullptr)) return 1;
    const size_t gbytes = static_cast<size_t>(h->num_envs) * (h->hm.task_kind >= dmk::kTaskHeadingGetup ? 4 : 3) * sizeof(float);
    DM_CUDA(cudaMemcpyAsync(h->p_goal, h->d_goal, gbytes, cudaMemcpyDeviceToHost, h->stream));
    DM_CUDA(cudaStreamSynchronize(h->stream));
    std::memcpy(h_out, h->p_goal, gbytes);
    return 0;
}
// test hooks of the task scenes: the environment's task block (dm_task.cuh: TaskSlot) and the scene constants as the device sees them
int dm_get_task_state(dm_handle* h, int env, double* h_out) {
    if (h->hm.task_kind == dmk::kTaskNone) { g_err = "dm_get_task_state: not a task scene"; return fail(); }
    DM_DEVICE(h);
    if (bad_env(h, env, "dm_get_task_state")) return fail();
    DM_CUDA(cudaStreamSynchronize(h->stream));
    DM_CUDA(cudaMemcpy(h_out, h->st.task + static_cast<size_t>(env) * dmk::kTaskDoubles, dmk::kTaskDoubles * sizeof(double), cudaMemcpyDeviceToHost));
    DM_CUDA(cudaMemcpy(h_out + dmk::kTaskDoubles, h->st.taskx + static_cast<size_t>(env) * dmk::kTaskExtDoubles, dmk::kTaskExtDoubles * sizeof(double), cudaMemcpyDeviceToHost));
    return 0;
}
int dm_set_task_state(dm_handle* h, int env, const double* h_in) {
    if (h->hm.task_kind == dmk::kTaskNone) { g_err = "dm_set_task_state: not a task scene"; return fail(); }
    DM_DEVICE(h);
    if (bad_env(h, env, "dm_set_task_state")) return fail();
    DM_CUDA(cudaStreamSynchronize(h->stream));
    DM_CUDA(cudaMemcpy(h->st.task + static_cast<size_t>(env) * dmk::kTaskDoubles, h_in, dmk::kTaskDoubles * sizeof(double), cudaMemcpyHostToDevice));
    DM_CUDA(cudaMemcpy(h->st.taskx + static_cast<size_t>(env) * dmk::kTaskExtDoubles, h_in + dmk::kTaskDoubles, dmk::kTaskExtDoubles * sizeof(double), cudaMemcpyHostToDevice));
    return 0;
}
int dm_get_task_params(dm_handle* h, double* o, unsigned long long* stream) {
    const dmk::TaskParams& T = h->hm.task;
    o[0] = h->hm.task_kind; o[1] = T.timer_min; o[2] = T.timer_max; o[3] = T.max_target_dist; o[4] = T.target_succ_dist; o[5] = T.tar_fail_dist; o[6] = T.pos_reward_scale;
    o[7] = T.max_heading_turn_rate; o[8] = T.sharp_turn_prob; o[9] = T.speed_change_prob; o[10] = T.tar_speed_min; o[11] = T.tar_speed_max; o[12] = T.vel_reward_scale;
    o[13] = T.tar_speed; o[14] = T.enable_min_tar_vel; o[15] = 0;
    {   // dm_task_ext.cuh constants, in the order tests/task_shim.cpp reads them
        const dmk::TaskExtParams& X = h->hm.taskx;
        double* q = o + 16;
        q[0] = X.getup_time; q[1] = X.getup_height_root; q[2] = X.getup_height_head; q[3] = X.recover_episode_prob;
        for (int k = 0; k < 3; ++k) { q[4 + k] = X.target_min[k]; q[7 + k] = X.target_max[k]; }
        q[10] = X.target_radius; q[11] = X.hit_reset_time; q[12] = X.tar_reward_scale; q[13] = X.hit_tar_speed; q[14] = X.init_hit_prob; q[15] = X.tar_far_prob; q[16] = X.tar_near_dist;
        q[17] = X.head_id; q[18] = X.n_strike; q[23] = X.n_fail;
        for (int k = 0; k < 4; ++k) { q[19 + k] = X.strike_bodies[k]; q[24 + k] = X.fail_bodies[k]; }
        q[28] = q[29] = q[30] = q[31] = 0;
    }
    if (stream) { stream[0] = h->hm.task_seed; stream[1] = h->hm.env_id_base; }
    return 0;
}
int dm_record_amp_obs_agent(dm_handle* h, float* d_out) { DM_DEVICE(h); return launch_amp(h, d_out, 0, nullptr); }
int dm_amp_obs_host(dm_handle* h, int expert, const double* h_kin_time, float* h_out) {
    DM_DEVICE(h);
    if (expert ? dm_record_amp_obs_expert(h, h_kin_time, h->d_amp) : dm_record_amp_obs_agent(h, h->d_amp)) return 1;
    const size_t bytes = static_cast<size_t>(h->num_envs) * h->hm.amp_obs_size * sizeof(float);
    DM_CUDA(cudaMemcpyAsync(h->p_amp, h->d_amp, bytes, cudaMemcpyDeviceToHost, h->stream));
    DM_CUDA(cudaStreamSynchronize(h->stream));
    std::memcpy(h_out, h->p_amp, bytes);
    return 0;
}
// host-side counter-based uniform for the expert draws (same finaliser as the device streams)
static double host_u01(unsigned long long seed, unsigned long long a, unsigned long long b) {
    unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (a * 2654435761ull + b + 1);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull; z = (z ^ (z >> 27)) * 0x94D049BB133111EBull; z ^= z >> 31;
    return static_cast<double>(z >> 11) * (1.0 / 9007199254740992.0);
}
int dm_record_amp_obs_expert_clips(dm_handle* h, const int* h_clip, const double* h_kin_time, float* d_out) {
    DM_DEVICE(h);
    const bool task = is_task(h);
    if (h_clip && !task) { g_err = "dm_record_amp_obs_expert_clips: clip ids can only be given in the AMP task scenes"; return fail(); }
    std::vector<double> tmp(h->padded_envs, 0.0);
    std::vector<int> ct(h->padded_envs, 0);
    if (task) {   // cSceneImitateAMP::SampleExpertMotion: cClipsController::SampleMotionID per call (SceneImitateAMP.cpp:260-277)
        for (int e = 0; e < h->num_envs; ++e) {
            ct[e] = h_clip ? h_clip[e] : dmk::select_clip(h->ctab, host_u01(h->seed ^ 0x657870636c6970ull, h->env_offset + e, h->amp_calls));
            if (ct[e] < 0 || ct[e] >= h->ctab.num_clips) { g_err = "dm_record_amp_obs_expert_clips: clip id out of range"; return fail(); }
        }
    }
    if (h_kin_time) std::copy(h_kin_time, h_kin_time + h->num_envs, tmp.begin());
    else {   // cSceneImitateAMP::RecordAMPObsExpert draws U(0, duration) per call; here a counter-based stream per (seed, env, call)
        for (int e = 0; e < h->num_envs; ++e) {
            const double dur = task ? h->ctab.info[ct[e]].dur : h->hm.motion_dur;
            tmp[e] = dur * host_u01(h->seed, h->env_offset + e, 0x51ed27ull + h->amp_calls - 1);
        }
    }
    if (!h_kin_time || (task && !h_clip)) h->amp_calls++;
    DM_CUDA(cudaMemcpyAsync(h->d_inj[0], tmp.data(), sizeof(double) * h->padded_envs, cudaMemcpyHostToDevice, h->stream));
    if (task) DM_CUDA(cudaMemcpyAsync(h->d_clip_inj, ct.data(), sizeof(int) * h->padded_envs, cudaMemcpyHostToDevice, h->stream));
    DM_CUDA(cudaStreamSynchronize(h->stream));   // tmp / ct are pageable host memory
    return launch_amp(h, d_out, 1, h->d_inj[0], task ? h->d_clip_inj : nullptr);
}
int dm_record_amp_obs_expert(dm_handle* h, const double* h_kin_time, float* d_out) { return dm_record_amp_obs_expert_clips(h, nullptr, h_kin_time, d_out); }
int dm_calc_reward(dm_handle* h, float* d_out) { return dm_observe(h, nullptr, d_out); }
int dm_get_flags(dm_handle* h, int32_t* d_flags) {
    DM_DEVICE(h);
    dmk::dm_flags_kernel<<<(h->num_envs + 127) / 128, 128, 0, h->stream>>>(h->st, d_flags, h->num_envs);
    return launched(h);
}
// true when the host pointer is page-locked (cudaMallocHost / cudaHostRegister): the copy engines can address it directly
static bool is_pinned_host(dm_handle* h, const void* p) {
    for (const auto& e : h->pin_cache) if (e.first == p) return e.second;
    cudaPointerAttributes at;
    bool pinned = false;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) cudaGetLastError();
    else pinned = at.type == cudaMemoryTypeHost;
    // a stale entry (buffer freed and the address reused with the other kind) costs performance only: cudaMemcpyAsync accepts pageable memory
    if (h->pin_cache.size() >= 32) h->pin_cache.clear();
    h->pin_cache.emplace_back(p, pinned);
    return pinned;
}
static inline double now_ms() {
    timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts);
    return 1e3 * static_cast<double>(ts.tv_sec) + 1e-6 * static_cast<double>(ts.tv_nsec);
}
int dm_set_timing(dm_handle* h, int on) {
    DM_DEVICE(h);
    if (on && !h->tev[0]) for (auto& e : h->tev) DM_CUDA(cudaEventCreate(&e));
    h->timing = on != 0;
    return 0;
}
int dm_step_host_timing(dm_handle* h, double* o) {
    DM_DEVICE(h);
    if (!h->timing || !h->tev[0]) { g_err = "dm_step_host_timing: call dm_set_timing(h, 1) before the dm_step_host to be measured"; return fail(); }
    float ms[4] = {0, 0, 0, 0};
    for (int k = 0; k < 4; ++k) DM_CUDA(cudaEventElapsedTime(&ms[k], h->tev[k], h->tev[k + 1]));
    for (int k = 0; k < 4; ++k) o[k] = ms[k];
    o[4] = h->host_ms[0]; o[5] = h->host_ms[1]; o[6] = h->host_ms[2]; o[7] = 0.0;
    return 0;
}
int dm_step_host(dm_handle* h, const float* h_actions, double dt, int n_updates, float* h_state, float* h_reward, int32_t* h_flags) {
    return dm_step_host_reset(h, h_actions, dt, n_updates, h_state, h_reward, h_flags, 0);
}
int dm_step_host_reset(dm_handle* h, const float* h_actions, double dt, int n_updates, float* h_state, float* h_reward, int32_t* h_flags, int reset_done) {
    DM_DEVICE(h);
    const size_t N = h->num_envs, A = h->hm.action_size, S = h->hm.state_size;
    // page-locked caller buffers are used as they are; pageable ones go through the handle's pinned staging buffers (one extra host copy)
    const bool pa = h_actions && is_pinned_host(h, h_actions), ps = h_state && is_pinned_host(h, h_state), pr = h_reward && is_pinned_host(h, h_reward),
               pf = h_flags && is_pinned_host(h, h_flags);
    const bool tm = h->timing;
    const double t0 = tm ? now_ms() : 0.0;
    double t_copy = 0.0;
    if (tm) DM_CUDA(cudaEventRecord(h->tev[0], h->stream));
    if (h_actions) {
        if (!pa) { const double c0 = tm ? now_ms() : 0.0; std::memcpy(h->p_act, h_actions, N * A * sizeof(float)); if (tm) t_copy += now_ms() - c0; }
        DM_CUDA(cudaMemcpyAsync(h->d_act, pa ? h_actions : h->p_act, N * A * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        if (dm_set_action(h, h->d_act)) return 1;
    }
    if (tm) DM_CUDA(cudaEventRecord(h->tev[1], h->stream));
    if (n_updates > 0 && dm_update(h, dt, n_updates)) return 1;
    if (tm) DM_CUDA(cudaEventRecord(h->tev[2], h->stream));
    if (dm_observe(h, h_state ? h->d_obs : nullptr, h_reward ? h->d_rew : nullptr)) return 1;
    if (h_flags && dm_get_flags(h, h->d_flags4)) return 1;
    if (tm) DM_CUDA(cudaEventRecord(h->tev[3], h->stream));
    if (h_state) DM_CUDA(cudaMemcpyAsync(ps ? h_state : h->p_obs, h->d_obs, N * S * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (h_reward) DM_CUDA(cudaMemcpyAsync(pr ? h_reward : h->p_rew, h->d_rew, N * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    if (h_flags) DM_CUDA(cudaMemcpyAsync(pf ? h_flags : h->p_flags, h->d_flags4, N * 4 * sizeof(int32_t), cudaMemcpyDeviceToHost, h->stream));
    if (tm) DM_CUDA(cudaEventRecord(h->tev[4], h->stream));
    const double t1 = tm ? now_ms() : 0.0;
    DM_CUDA(cudaStreamSynchronize(h->stream));
    const double t2 = tm ? now_ms() : 0.0;
    if (h_state && !ps) std::memcpy(h_state, h->p_obs, N * S * sizeof(float));
    if (h_reward && !pr) std::memcpy(h_reward, h->p_rew, N * sizeof(float));
    if (h_flags && !pf) std::memcpy(h_flags, h->p_flags, N * 4 * sizeof(int32_t));
    if (tm) { h->host_ms[0] = t1 - t0 - t_copy; h->host_ms[1] = t2 - t1; h->host_ms[2] = t_copy + (now_ms() - t2); }
    // the caller has the finished episodes' last state / reward / flags: restart them now, after the wait, so that the reset kernel runs
    // under the caller's own work and the next call finds the stream idle (the reference's caller resets right after IsEpisodeEnd)
    if (reset_done) return dm_reset(h, 0, nullptr, nullptr, nullptr);
    return 0;
}

// ---------------------------------------------------------------- multi-GPU exchange over NVLink peer memory (include/deepmimic_b200.h)
static size_t xchg_parity_floats(const dm_handle* h) { return static_cast<size_t>(h->x_world) * h->num_envs * (h->hm.state_size + 2); }
static float* xchg_plane(const dm_handle* h, const char* base, int parity, int plane /*0 obs 1 rew 2 done*/) {
    const size_t WN = static_cast<size_t>(h->x_world) * h->num_envs, S = h->hm.state_size;
    float* p = reinterpret_cast<float*>(const_cast<char*>(base) + h->x_data_off + static_cast<size_t>(parity) * h->x_parity_bytes);
    return plane == 0 ? p : (plane == 1 ? p + WN * S : p + WN * S + WN);
}
int dm_exchange_create(dm_handle* h, int rank, int world, void* h_ipc_out64) {
    DM_DEVICE(h);
    if (h->x_base) { g_err = "dm_exchange_create: the handle already has an exchange"; return fail(); }
    if (world < 1 || world > 8 || rank < 0 || rank >= world) { g_err = "dm_exchange_create: world must be 1..8 (one node) and 0 <= rank < world"; return fail(); }
    h->x_rank = rank; h->x_world = world;
    h->x_data_off = 1024;
    h->x_parity_bytes = ((xchg_parity_floats(h) * sizeof(float) + 255) / 256) * 256;
    const size_t bytes = h->x_data_off + 2 * h->x_parity_bytes;
    DM_CUDA(cudaMalloc(&h->x_base, bytes));
    DM_CUDA(cudaMemset(h->x_base, 0, bytes));
    DM_CUDA(cudaDeviceSynchronize());
    h->x_peer[rank] = h->x_base;
    cudaIpcMemHandle_t ipc;
    DM_CUDA(cudaIpcGetMemHandle(&ipc, h->x_base));
    static_assert(sizeof(ipc) == 64, "cudaIpcMemHandle_t is 64 bytes");
    std::memcpy(h_ipc_out64, &ipc, 64);
    return 0;
}
int dm_exchange_connect(dm_handle* h, const void* h_ipc_all) {
    DM_DEVICE(h);
    if (!h->x_base) { g_err = "dm_exchange_connect: call dm_exchange_create first"; return fail(); }
    for (int r = 0; r < h->x_world; ++r) {
        if (r == h->x_rank) continue;
        cudaIpcMemHandle_t ipc;
        std::memcpy(&ipc, static_cast<const char*>(h_ipc_all) + 64 * r, 64);
        void* p = nullptr;
        DM_CUDA(cudaIpcOpenMemHandle(&p, ipc, cudaIpcMemLazyEnablePeerAccess));
        h->x_peer[r] = static_cast<char*>(p);
    }
    return 0;
}
static dmk::XchgPeers xchg_peers(const dm_handle* h) {
    dmk::XchgPeers P{};
    P.n = h->x_world;
    for (int r = 0; r < h->x_world; ++r) P.f[r] = reinterpret_cast<dmk::XchgFlags*>(h->x_peer[r]);
    return P;
}
static const unsigned long long kXchgTimeoutNs = 20ull * 1000ull * 1000ull * 1000ull;
int dm_exchange_publish(dm_handle* h, long long step) {
    DM_DEVICE(h);
    if (!h->x_base) { g_err = "dm_exchange_publish: no exchange (dm_exchange_create / dm_exchange_connect)"; return fail(); }
    for (int r = 0; r < h->x_world; ++r) if (!h->x_peer[r]) { g_err = "dm_exchange_publish: peers are not connected"; return fail(); }
    if (is_task(h)) { g_err = "dm_exchange_publish: the AMP task scenes are not wired to the exchange"; return fail(); }
    const int par = static_cast<int>(step & 1);
    if (step >= 2 && h->x_world > 1) {   // the slot still holds step - 2: every rank must have released it
        dmk::dm_xchg_wait_kernel<<<1, 32, 0, h->stream>>>(reinterpret_cast<dmk::XchgFlags*>(h->x_base), h->x_world, 1, static_cast<unsigned long long>(step - 1), kXchgTimeoutNs);
        if (launched(h)) return 1;
    }
    dmk::ObsFan fan{};
    fan.n = h->x_world;
    const size_t N = h->num_envs, S = h->hm.state_size;
    int d = 0;
    for (int k = 0; k < h->x_world; ++k) {   // destination 0 = local, then the peers starting after this rank (spreads the first stores over the links)
        const int r = (h->x_rank + k) % h->x_world;
        fan.obs[d] = xchg_plane(h, h->x_peer[r], par, 0) + h->x_rank * N * S;
        fan.rew[d] = xchg_plane(h, h->x_peer[r], par, 1) + h->x_rank * N;
        fan.done[d] = xchg_plane(h, h->x_peer[r], par, 2) + h->x_rank * N;
        ++d;
    }
    if (launch_observe_fan(h, fan)) return 1;
    dmk::dm_xchg_signal_kernel<<<1, 32, 0, h->stream>>>(xchg_peers(h), h->x_rank, 0, static_cast<unsigned long long>(step + 1));
    return launched(h);
}
int dm_exchange_acquire(dm_handle* h, long long step, float** d_obs, float** d_rew, float** d_done) {
    DM_DEVICE(h);
    if (!h->x_base) { g_err = "dm_exchange_acquire: no exchange"; return fail(); }
    if (h->x_world > 1) {
        dmk::dm_xchg_wait_kernel<<<1, 32, 0, h->stream>>>(reinterpret_cast<dmk::XchgFlags*>(h->x_base), h->x_world, 0, static_cast<unsigned long long>(step + 1), kXchgTimeoutNs);
        if (launched(h)) return 1;
    }
    const int par = static_cast<int>(step & 1);
    if (d_obs) *d_obs = xchg_plane(h, h->x_base, par, 0);
    if (d_rew) *d_rew = xchg_plane(h, h->x_base, par, 1);
    if (d_done) *d_done = xchg_plane(h, h->x_base, par, 2);
    return 0;
}
int dm_exchange_release(dm_handle* h, long long step) {
    DM_DEVICE(h);
    if (!h->x_base) { g_err = "dm_exchange_release: no exchange"; return fail(); }
    if (h->x_world > 1) {
        dmk::dm_xchg_signal_kernel<<<1, 32, 0, h->stream>>>(xchg_peers(h), h->x_rank, 1, static_cast<unsigned long long>(step + 1));
        if (launched(h)) return 1;
    }
    return 0;
}
int dm_exchange_status(dm_handle* h, int* status) {
    DM_DEVICE(h);
    if (!h->x_base) { g_err = "dm_exchange_status: no exchange"; return fail(); }
    DM_CUDA(cudaStreamSynchronize(h->stream));
    unsigned int s = 0;
    DM_CUDA(cudaMemcpy(&s, h->x_base + offsetof(dmk::XchgFlags, status), sizeof(s), cudaMemcpyDeviceToHost));
    *status = static_cast<int>(s);
    return 0;
}
int dm_exchange_destroy(dm_handle* h) {
    if (!h->x_base) return 0;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    for (int r = 0; r < h->x_world; ++r) if (r != h->x_rank && h->x_peer[r]) { cudaIpcCloseMemHandle(h->x_peer[r]); }
    for (auto& p : h->x_peer) p = nullptr;
    cudaFree(h->x_base); h->x_base = nullptr; h->x_world = 0;
    return 0;
}

int dm_get_snapshot(dm_handle* h, int env, double* s) {
    DM_DEVICE(h);
    if (bad_env(h, env, "dm_get_snapshot")) return fail();
    const auto& M = h->hm; const int nl = M.nl, ss = dmk::sim_stride(nl);
    std::vector<float> sim(ss), man(nl * dmk::kManifoldFloats); double tm[dmk::kTimeDoubles]; int fl[dmk::kFlagInts];
    DM_CUDA(cudaStreamSynchronize(h->stream));
    DM_CUDA(cudaMemcpy(sim.data(), h->st.sim + static_cast<size_t>(env) * ss, ss * sizeof(float), cudaMemcpyDeviceToHost));
    DM_CUDA(cudaMemcpy(man.data(), h->st.manifold + static_cast<size_t>(env) * nl * dmk::kManifoldFloats, man.size() * sizeof(float), cudaMemcpyDeviceToHost));
    DM_CUDA(cudaMemcpy(tm, h->st.time + static_cast<size_t>(env) * dmk::kTimeDoubles, sizeof(tm), cudaMemcpyDeviceToHost));
    DM_CUDA(cudaMemcpy(fl, h->st.flags + static_cast<size_t>(env) * dmk::kFlagInts, sizeof(fl), cudaMemcpyDeviceToHost));
    std::fill(s, s + 29 + 59 * nl, 0.0);
    for (int k = 0; k < 3; ++k) { s[k] = sim[k]; s[7 + k] = sim[8 + k]; s[10 + k] = sim[12 + k]; }
    for (int k = 0; k < 4; ++k) s[3 + k] = sim[4 + k];
    for (int j = 0; j < nl; ++j) {
        if (M.link[j].ndof > 0) for (int k = 0; k < 4; ++k) s[13 + 4 * j + k] = sim[16 + 4 * j + k];
        else s[13 + 4 * j + 3] = 1.0;
        for (int k = 0; k < M.link[j].ndof; ++k) s[13 + 4 * nl + 3 * j + k] = sim[16 + 4 * nl + 4 * j + k];
        for (int c = 0; c < 4; ++c) for (int k = 0; k < 12; ++k) s[13 + 7 * nl + (j * 4 + c) * 12 + k] = man[j * dmk::kManifoldFloats + c * 12 + k];
        // PD target back to the joint-frame (w,x,y,z) convention
        const float* t = &sim[16 + 8 * nl + 4 * j]; double* o = s + 29 + 55 * nl + 4 * j;
        if (M.link[j].jtype == dmk::kJSpherical) {
            Quat cr(M.link[j].child_rot[3], M.link[j].child_rot[0], M.link[j].child_rot[1], M.link[j].child_rot[2]);
            Quat q = dmh::conj(cr) * Quat(t[3], t[0], t[1], t[2]) * cr;
            o[0] = q.w; o[1] = q.x; o[2] = q.y; o[3] = q.z;
        } else if (M.link[j].jtype == dmk::kJRevolute) o[0] = t[0];
    }
    double* q = s + 13 + 55 * nl;
    q[0] = tm[dmk::kTKin]; q[1] = tm[dmk::kTOrigin]; q[2] = tm[dmk::kTOrigin + 1]; q[3] = tm[dmk::kTOrigin + 2];
    for (int k = 0; k < 4; ++k) q[4 + k] = tm[dmk::kTOriginRot + k];
    q[8] = tm[dmk::kTCtrl]; q[9] = tm[dmk::kTInitOff]; q[10] = tm[dmk::kTPrevAct]; q[11] = fl[dmk::kFNeedAction]; q[12] = tm[dmk::kTTimer]; q[13] = tm[dmk::kTTimerMax];
    return 0;
}
int dm_set_snapshot(dm_handle* h, int env, const double* s) {
    DM_DEVICE(h);
    if (bad_env(h, env, "dm_set_snapshot")) return fail();
    const auto& M = h->hm; const int nl = M.nl, ss = dmk::sim_stride(nl);
    std::vector<float> sim(ss, 0.f), man(nl * dmk::kManifoldFloats, 0.f); double tm[dmk::kTimeDoubles] = {0}; int fl[dmk::kFlagInts] = {0};
    DM_CUDA(cudaStreamSynchronize(h->stream));
    DM_CUDA(cudaMemcpy(fl, h->st.flags + static_cast<size_t>(env) * dmk::kFlagInts, sizeof(fl), cudaMemcpyDeviceToHost));
    for (int k = 0; k < 3; ++k) { sim[k] = static_cast<float>(s[k]); sim[8 + k] = static_cast<float>(s[7 + k]); sim[12 + k] = static_cast<float>(s[10 + k]); }
    for (int k = 0; k < 4; ++k) sim[4 + k] = static_cast<float>(s[3 + k]);
    for (int j = 0; j < nl; ++j) {
        for (int k = 0; k < 4; ++k) sim[16 + 4 * j + k] = static_cast<float>(s[13 + 4 * j + k]);
        for (int k = 0; k < M.link[j].ndof; ++k) sim[16 + 4 * nl + 4 * j + k] = static_cast<float>(s[13 + 4 * nl + 3 * j + k]);
        for (int c = 0; c < 4; ++c) for (int k = 0; k < 12; ++k) man[j * dmk::kManifoldFloats + c * 12 + k] = static_cast<float>(s[13 + 7 * nl + (j * 4 + c) * 12 + k]);
        const double* o = s + 29 + 55 * nl + 4 * j; float* t = &sim[16 + 8 * nl + 4 * j];
        if (M.link[j].jtype == dmk::kJSpherical) {
            Quat cr(M.link[j].child_rot[3], M.link[j].child_rot[0], M.link[j].child_rot[1], M.link[j].child_rot[2]);
            Quat q = cr * Quat(o[0], o[1], o[2], o[3]) * dmh::conj(cr);
            t[0] = static_cast<float>(q.x); t[1] = static_cast<float>(q.y); t[2] = static_cast<float>(q.z); t[3] = static_cast<float>(q.w);
        } else if (M.link[j].jtype == dmk::kJRevolute) t[0] = static_cast<float>(o[0]);
    }
    const double* q = s + 13 + 55 * nl;
    tm[dmk::kTKin] = q[0]; tm[dmk::kTOrigin] = q[1]; tm[dmk::kTOrigin + 1] = q[2]; tm[dmk::kTOrigin + 2] = q[3];
    for (int k = 0; k < 4; ++k) tm[dmk::kTOriginRot + k] = q[4 + k];
    tm[dmk::kTCtrl] = q[8]; tm[dmk::kTInitOff] = q[9]; tm[dmk::kTPrevAct] = q[10]; tm[dmk::kTTimer] = q[12]; tm[dmk::kTTimerMax] = q[13];
    fl[dmk::kFNeedAction] = q[11] != 0; fl[dmk::kFDone] = 0; fl[dmk::kFTerminate] = 0; fl[dmk::kFValid] = 1; fl[dmk::kFFallen] = 0;
    DM_CUDA(cudaMemcpy(h->st.sim + static_cast<size_t>(env) * ss, sim.data(), ss * sizeof(float), cudaMemcpyHostToDevice));
    DM_CUDA(cudaMemcpy(h->st.manifold + static_cast<size_t>(env) * nl * dmk::kManifoldFloats, man.data(), man.size() * sizeof(float), cudaMemcpyHostToDevice));
    DM_CUDA(cudaMemcpy(h->st.time + static_cast<size_t>(env) * dmk::kTimeDoubles, tm, sizeof(tm), cudaMemcpyHostToDevice));
    DM_CUDA(cudaMemcpy(h->st.flags + static_cast<size_t>(env) * dmk::kFlagInts, fl, sizeof(fl), cudaMemcpyHostToDevice));
    return 0;
}
int dm_debug_enable(dm_handle* h, int on) {
    DM_DEVICE(h);
    DM_CUDA(cudaStreamSynchronize(h->stream));
    if (on && !h->st.pdbg) {
        DM_CUDA(cudaMalloc(&h->st.pdbg, static_cast<size_t>(h->padded_envs) * dmk::kDebugFloats * sizeof(float)));
        DM_CUDA(cudaMemset(h->st.pdbg, 0, static_cast<size_t>(h->padded_envs) * dmk::kDebugFloats * sizeof(float)));
    } else if (!on && h->st.pdbg) { cudaFree(h->st.pdbg); h->st.pdbg = nullptr; }
    return 0;
}
int dm_get_debug(dm_handle* h, int env, float* out) {
    DM_DEVICE(h);
    if (bad_env(h, env, "dm_get_debug")) return fail();
    DM_CUDA(cudaStreamSynchronize(h->stream));
    if (!h->st.pdbg) { g_err = "debug dumps are not enabled"; return fail(); }
    DM_CUDA(cudaMemcpy(out, h->st.pdbg + static_cast<size_t>(env) * dmk::kDebugFloats, dmk::kDebugFloats * sizeof(float), cudaMemcpyDeviceToHost));
    return 0;
}
int dm_get_counters(dm_handle* h, int64_t* out) {
    DM_DEVICE(h);
    DM_CUDA(cudaStreamSynchronize(h->stream));
    std::vector<int> fl(static_cast<size_t>(h->padded_envs) * dmk::kFlagInts);
    DM_CUDA(cudaMemcpy(fl.data(), h->st.flags, fl.size() * sizeof(int), cudaMemcpyDeviceToHost));
    int64_t over = 0;
    for (int e = 0; e < h->num_envs; ++e) over += fl[static_cast<size_t>(e) * dmk::kFlagInts + dmk::kFRowOverflow];
    out[0] = h->launches; out[1] = over;
    return 0;
}

}  // extern "C"
