// Fused per-update kernel (articulated-body formulation): one launch advances every environment by n_updates x Update(dt),
// i.e. per update exactly what the reference does in cSceneSimChar::Update (R/DeepMimicCore/scenes/SceneSimChar.cpp:136-161):
//   kin clock / cycle sync  (scenes/SceneImitate.cpp:306-318,420-444)
//   Stable-PD torques       (sim/ImpPDController.cpp:136-195): (M + dt Kd) a = Kp e + Kd edot - C, tau = Kp e + Kd (edot - dt a)
//   2 x Bullet sub-step     (sim/World.cpp:93-104): link-vs-plane manifolds, Featherstone forward dynamics, contact / friction /
//                           joint-limit rows, 10 projected-Gauss-Seidel sweeps, exponential-map integration
//   controller clock + 30 Hz "need action" edge (sim/CtController.cpp:221-227), fall / explode / timer flags.
//
// B200 mapping: one tile of W lanes (16 or 32) per environment, lane = link.  Every linear solve with the joint-space mass
// matrix is done by the articulated-body recursion (the tree-structured L^T D L factorisation in its O(depth) form): one
// leaves->root pass builds articulated inertias in registers (a link publishes its shifted inertia in shared scratch, its parent
// adds its children's), one root->leaves pass propagates accelerations; both run on a dynamics tree without the dof-less links
// (root referred to the base origin, fixed leaves lumped into their parents).  The Stable-PD system is the same recursion with
// dt*Kd added to the joint-space diagonal and DeepMimic's exact-shape inertias; the Bullet sub-steps use Bullet's collision-shape
// inertias (their unconstrained accelerations are btMultiBody::computeAccelerationsArticulatedBodyAlgorithmMultiDof's).
// Constraint rows are built with lanes = rows (each lane walks its row's link chain once), the row coupling matrix
// J M^-1 J^T is formed explicitly in shared memory with lanes = pairs of contact points (3 x 3 blocks), and PGS runs in impulse
// space: w = A lambda lives in registers (lane = row), the sequential sweep is evaluated in blocks of two solver steps by every lane
// redundantly from broadcast row data (the figure of merit is warp instructions per step: the sweeps are issue-bound).
// All spatial quantities of a link are expressed in WORLD axes about the link's own joint pivot, so passing them between
// parent and child is a pure shift (no rotation of 6x6 blocks).
// The update is split into phase routines (kinematics, collision, articulated-body solve, constraint rows + PGS, velocity correction)
// that are deliberately NOT inlined: they exchange state through the environment's shared-memory block, so each phase gets the full
// register budget and the main loop only carries the joint state of its link.  The warps of a block run in lockstep (a barrier after
// every stage: the ~9 k-instruction loop does not fit the instruction cache otherwise), which makes every unconditional memory burst a
// contention point: the collision routine touches a link's persistent manifold only when it can matter.
// No tensor cores: there is no dense contraction here (34 or 70 dofs, tree-sparse); the path is latency-bound.
#include "dm_model.cuh"
#include <type_traits>

namespace dmk {

namespace {

template <int W>
struct Tl {
    static __device__ __forceinline__ float shfl(float v, int src) { return __shfl_sync(0xffffffffu, v, src, W); }
    static __device__ __forceinline__ int shfli(int v, int src) { return __shfl_sync(0xffffffffu, v, src, W); }
    static __device__ __forceinline__ V3 shfl3(V3 v, int src) { return mk3(shfl(v.x, src), shfl(v.y, src), shfl(v.z, src)); }
    static __device__ __forceinline__ S6 shfl6(S6 v, int src) { return mks(shfl3(v.a, src), shfl3(v.l, src)); }
};
// 12-float shared-memory records (48 bytes, 16-byte aligned: every offset of the environment block is a multiple of 4 floats) move as three 128-bit accesses
__device__ __forceinline__ void ld12(const float* p, float* o) {
    const float4 a = reinterpret_cast<const float4*>(p)[0], b = reinterpret_cast<const float4*>(p)[1], c_ = reinterpret_cast<const float4*>(p)[2];
    o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w; o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w; o[8] = c_.x; o[9] = c_.y; o[10] = c_.z; o[11] = c_.w;
}
__device__ __forceinline__ void st12(float* p, const float* o) {
    reinterpret_cast<float4*>(p)[0] = make_float4(o[0], o[1], o[2], o[3]); reinterpret_cast<float4*>(p)[1] = make_float4(o[4], o[5], o[6], o[7]);
    reinterpret_cast<float4*>(p)[2] = make_float4(o[8], o[9], o[10], o[11]);
}
__device__ __forceinline__ float rcp_fast(float x) { float r; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x)); return r; }
__device__ __forceinline__ int wmax(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = max(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}

// articulated (or rigid) spatial inertia about a link's joint pivot, world axes:  n = ww*w + wv*v ; f = wv^T*w + vv*v
struct Art {
    float ww[6];   // xx xy xz yy yz zz
    float wv[9];   // row major
    float vv[6];
};
__device__ __forceinline__ V3 wvT_mul(const float* g, V3 w) { return mk3(g[0] * w.x + g[3] * w.y + g[6] * w.z, g[1] * w.x + g[4] * w.y + g[7] * w.z, g[2] * w.x + g[5] * w.y + g[8] * w.z); }
// R^T S R for a symmetric S (R row-major, maps parent -> child axes)
__device__ __forceinline__ void rot_sym(const M3& R, const float* s, float* o) {
    // T = S R (3x3), o = R^T T (symmetric)
    float t[9];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        t[0 + j] = s[0] * R.m[j] + s[1] * R.m[3 + j] + s[2] * R.m[6 + j];
        t[3 + j] = s[1] * R.m[j] + s[3] * R.m[3 + j] + s[4] * R.m[6 + j];
        t[6 + j] = s[2] * R.m[j] + s[4] * R.m[3 + j] + s[5] * R.m[6 + j];
    }
    o[0] = R.m[0] * t[0] + R.m[3] * t[3] + R.m[6] * t[6];
    o[1] = R.m[0] * t[1] + R.m[3] * t[4] + R.m[6] * t[7];
    o[2] = R.m[0] * t[2] + R.m[3] * t[5] + R.m[6] * t[8];
    o[3] = R.m[1] * t[1] + R.m[4] * t[4] + R.m[7] * t[7];
    o[4] = R.m[1] * t[2] + R.m[4] * t[5] + R.m[7] * t[8];
    o[5] = R.m[2] * t[2] + R.m[5] * t[5] + R.m[8] * t[8];
}
__device__ __forceinline__ float normalize_angle3(float t) {  // cMathUtil::NormalizeAngle
    float n = fmodf(t, 6.283185307179586f);
    if (n > 3.14159265358979f) n -= 6.283185307179586f;
    else if (n < -3.14159265358979f) n += 6.283185307179586f;
    return n;
}
// rotation vector of a unit quaternion, same semantics as cMathUtil::QuaternionToAxisAngle (theta in [-pi,pi], zero when
// sin(theta/2) <= 1e-6) but evaluated with atan2 so small angles keep fp32 accuracy
__device__ __forceinline__ V3 quat_rotvec3(Q4 q) {
    float s = sqrtf(q.x * q.x + q.y * q.y + q.z * q.z);
    if (!(s > 0.000001f)) return mk3(0.f, 0.f, 0.f);
    float th = normalize_angle3(2.0f * atan2f(s, q.w));
    float k = th / s;
    return mk3(q.x * k, q.y * k, q.z * k);
}
// btMultiBody::stepPositionsMultiDof's exponential-map quaternion update
__device__ __forceinline__ Q4 quat_integrate3(V3 omega, Q4 quat, bool base_body, float dt) {
    V3 angvel = base_body ? omega : qrot(quat, omega);
    float fAngle = sqrtf(dot(angvel, angvel));
    const float kThr = 0.5f * 1.57079632679489661923f;
    if (fAngle * dt > kThr) fAngle = kThr / dt;
    V3 axis;
    if (fAngle < 0.001f) axis = angvel * (0.5f * dt - (dt * dt * dt) * 0.020833333333f * fAngle * fAngle);
    else axis = angvel * (__sinf(0.5f * fAngle * dt) / fAngle);   // |angle| <= pi/8 (ANGULAR_MOTION_THRESHOLD): fast path error ~1e-7
    float cw = __cosf(fAngle * dt * 0.5f);
    Q4 r = base_body ? qmul(quat, mkq(-axis.x, -axis.y, -axis.z, cw)) : qmul(mkq(axis.x, axis.y, axis.z, cw), quat);
    float n = rsqrtf(r.x * r.x + r.y * r.y + r.z * r.z + r.w * r.w);
    return mkq(r.x * n, r.y * n, r.z * n, r.w * n);
}

// ---- block-shared model table, floats per link (LK)
// (groups of four: the hot routines read a group with one 128-bit load)
enum LkSlot { kLC = 0 /*3*/, kLM = 3,                 // parent pivot -> pivot (parent axes) | own mass
              kLD = 4 /*3*/, kLThr = 7,               // pivot -> COM (link axes) | contact breaking threshold
              kLWd = 8 /*6*/, kLInt = 14 /* parent|jtype|ndof|depth0 */, kLInt2 = 15 /* dof0|lastd|nchild */,
              kLWb = 16 /*6*/, kLFlg = 22 /* shape | fall<<8 | has_limit<<16 */, kLTree = 23 /* level | maxlevel<<8 | nchild<<16 */,
              kLAx = 24 /*3*/, kLTl = 27,
              kLZr = 28 /*4*/,
              kLHe = 32 /*3*/, kLKp = 35,
              kLKd = 36, kLLo = 37, kLHi = 38, kLChild = 39 /* child lanes, 8 bits each */,
              kLDc = 40 /*3: reference point -> composite COM, link axes */, kLMc = 43 /* composite mass */,
              kLDyn = 44 /* dynamics tree: parent | level<<8 (signed: root -1, lumped 100) | bypassed kinematic parent<<16 (0xff none) | children<<24 */, kLDChild = 45 /* dynamics children, 8 bits each */,
              kLkFloats = 48 };
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
// ---- block-shared header in front of the link table (floats): the launch's StepLayout (24 ints), children per tree level (8 ints), constants
enum HdrSlot { kHLayout = 0, kHLvc = 24, kHGrav = 32 /*3*/, kHh = 35, kHScale = 36, kHMu = 37, kHFdt = 38, kHDmax = 39 /* int: deepest level of the dynamics tree */, kHdrFloats = 40 };
__device__ __forceinline__ float* step_smem() { extern __shared__ __align__(16) float dm_step_sm[]; return dm_step_sm; }

}  // namespace

int dm_step_layout(int nl, int n, int chain_len, int maxrows, int W, StepLayout* L) {
    const int maxpts = maxrows / 3;
    int o = 0;
    L->nl = nl; L->n = n; L->chain_len = chain_len; L->maxrows = maxrows; L->maxpts = maxpts;
    L->oU = o; o += nl * 24;                       // per link: U0 U1 U2 (6 each), 1/D (3), sqrt(1/D) (3)
    L->oR = o; o += nl * 12;                       // per link: joint axes in world axes (9), parent pivot -> pivot (3)
    L->oA = o;                                     // union { world frames + link velocities | packed lower triangle of J M^-1 J^T }
    const int world = nl * 24, tri = maxrows * (maxrows + 1) / 2;   // world: Rwl 9 + pivot 3 | link velocity 6 + pivot->COM 3 (+3 pad)
    L->oW = o; L->oV = o + nl * 12;
    o += (world > tri ? world : tri);
    o = (o + 3) & ~3;                              // 16-byte aligned: the articulated-body pass borrows the block as float4 scratch (28 floats per lane)
    const int ys = dm_step_y_stride(W);
    L->oY = o; o += (chain_len * ys > 28 * W) ? chain_len * ys : 28 * W;   // Yt[depth][row], row stride = the tile width's row capacity (a compile-time constant of the kernel: immediate offsets)
    L->oLam = o; o += maxrows; o += (o & 1); L->oRhs = o; o += maxrows; L->oInv = o; o += maxrows;   // oRhs .. : interleaved (rhs, 1 / A_ii) pairs, 8-byte aligned
    L->oRl = o; o += maxrows;                      // row -> link (int)
    L->oPp = o; o += maxpts * 4; L->oPi = o; o += maxpts; L->oPr = o; o += maxpts;
    L->oQ = o; o += 4 * 8;                         // limit rows: link, dir, penetration, joint rate (<= 8)
    L->oG = o; o += 21 + 13 + 2;                   // base Cholesky factor (21), base state: position 3, quaternion 4, omega 3, velocity 3
    L->oZ = o; o += ((n + 3) / 4) * 4;
    L->env_floats = ((o + 15) / 32) * 32 + 16;     // stride == 16 (mod 32 banks): the two environments of a warp (W = 16) hit disjoint bank halves
    L->hot_floats = kHdrFloats + ((nl * kLkFloats + (nl * nl + nl * chain_len + 3) / 4 + 3) / 4) * 4;
    return L->hot_floats * 4 + 0;
}
int dm_step_smem_bytes(const StepLayout& L, int tiles) { return (L.hot_floats + L.env_floats * tiles) * static_cast<int>(sizeof(float)); }

// Projected Gauss-Seidel in impulse space, 10 sweeps in btMultiBodyConstraintSolver::solveSingleIteration's row order (joint limits in
// alternating order, contact normals, friction pairs).  Lanes = rows for the state that is wide: every lane keeps w = (A lambda)_row of ITS rows in
// registers (S rows per lane: row = lane + s W).  The sequential part is evaluated in blocks of B consecutive solver steps of one section:
//     B independent shuffles fetch the block's w values from their owners; the rows' right-hand side, 1 / A_ii and impulse are broadcast loads,
//     EVERY lane then evaluates the B sequential Gauss-Seidel updates redundantly (row k+1 sees row k's update through A(k+1, k), B (B-1) / 2
//     broadcast entries of A), one lane per row commits the new impulse to shared memory,
//     and every lane adds A(own row, row_k) * delta_k, k = 0..B-1 in order, to its own w's.
// During the sweeps the warps of a block are issue-bound (3.5 warps per scheduler all inside this loop), so the figure of merit is warp
// instructions per solver step: ~40 with one shuffle per step (the owner computed and broadcast its update), ~20 here.  Every floating-point
// operation on w and the update, and their order, are those of the row-by-row sweep (resolveSingleConstraintRowGeneric: delta = rhs - w *
// jacDiagABInv, clamped sum; friction bounds +-mu * the point's current normal impulse, row skipped while that is <= 0).  Bounds are applied to
// the UPDATE: clamp(delta, lo - lambda, hi - lambda) equals Bullet's "clamp the sum, then delta = limit - applied" in every branch; the stored
// impulse is clamp(lambda + delta, lo, hi) (Bullet stores the limit itself when clamped: equal up to one rounding of lambda + (limit - lambda)).
// The two environments of a W = 16 warp run in lockstep, each with its own row numbering (shuffles are tile-wide).
// A: symmetric square of stride ST (W when the environment has at most W rows, kSq2 for up to kSq2 rows on two slots), packed lower triangle beyond.  sRI: (rhs, 1 / A_ii) pairs.  NLmax / Pmax: warp-wide maxima of NL / P
// (block loops are warp-uniform).
enum PgsSection { kSecLimit = 0, kSecNormal = 1, kSecFriction = 2 };
template <int W, int S, int ST, int B>   // ST > 0: A is a full symmetric square of stride ST; ST == 0: packed lower triangle
__device__ __forceinline__ void pgs_sweeps(const float* sA, float* sLam, const float2* sRI, int lane, int NL, int P, int NLmax, int Pmax, float mu) {
    using T = Tl<W>;
    float w[S];
#pragma unroll
    for (int s = 0; s < S; ++s) w[s] = 0.f;
    // A(lane + s W, i).  Lanes without a row read finite leftovers of the scratch region: their w is never fetched.  Packed storage: tri(r) = r (r + 1) / 2
    // of the lane's own rows is computed once, tri(i) once per solver step.
    int tjs[S];
#pragma unroll
    for (int s = 0; s < S; ++s) { const int rid = lane + s * W; tjs[s] = rid * (rid + 1) / 2; }
    auto tri = [](int i) { return (i * (i + 1)) >> 1; };
    auto a_own = [&](int s, int i, int ti) -> float {
        if (ST > 0) return sA[i * ST + lane + s * W];
        const int rid = lane + s * W;
        return sA[(rid >= i) ? (tjs[s] + i) : (ti + rid)];
    };
    auto a_pair = [&](int i, int j, int ti, int tj_) -> float {   // A(i, j), tile-uniform indices
        if (ST > 0) return sA[i * ST + j];
        return sA[(i >= j) ? (ti + j) : (tj_ + i)];
    };
    // warm start: w = A lambda0 (normals carry 0.85 x the cached impulse, everything else starts at 0), in point order
#pragma unroll 1
    for (int p = 0; p < Pmax; ++p) {
        const int i = NL + ((p < P) ? p : 0);
        const float l0 = (p < P) ? sLam[i] : 0.f;
#pragma unroll
        for (int s = 0; s < S; ++s) w[s] = fmaf(a_own(s, i, tri(i)), l0, w[s]);
    }
    bool writer[B];   // lane k of the tile commits the impulse of the block's k-th step
#pragma unroll
    for (int k = 0; k < B; ++k) writer[k] = lane == k;
    // one block of B consecutive solver steps of section SEC, starting at position pos0 of the section
    auto block = [&](int pos0, int it, auto sec_tag) {
        constexpr int SEC = decltype(sec_tag)::value;
        int ik[B], tk[B]; bool vk[B];
        float tot = 0.f;
        float wk[B], rhs[B], inv[B], lam[B], lo[B], hi[B], ain[B * (B - 1) / 2 > 0 ? B * (B - 1) / 2 : 1], ao[S][B];
        if (SEC == kSecLimit) {
#pragma unroll
            for (int k = 0; k < B; ++k) { const int pos = pos0 + k; vk[k] = pos < NL; ik[k] = vk[k] ? ((it & 1) ? pos : NL - 1 - pos) : 0; }
        } else {
            // normals / friction rows are consecutive: one base index, immediate offsets.  Steps past the section's end (the other environment of
            // the warp has more rows, or an odd count) keep their natural index: they read initialised words of the environment block (zeroed
            // at kernel start, see dm_step_kernel) and their update is forced to 0 below.
            const int i0 = ((SEC == kSecNormal) ? NL : NL + P) + pos0, cnt = (SEC == kSecNormal) ? P : 2 * P;
#pragma unroll
            for (int k = 0; k < B; ++k) { ik[k] = i0 + k; vk[k] = pos0 + k < cnt; }
        }
#pragma unroll
        for (int k = 0; k < B; ++k) tk[k] = (ST > 0) ? 0 : tri(ik[k]);
#pragma unroll
        for (int k = 0; k < B; ++k) {
            const float2 ri = sRI[ik[k]];
            rhs[k] = ri.x; inv[k] = ri.y; lam[k] = sLam[ik[k]];
            if (SEC == kSecFriction) {
                // the point's normal impulse of this sweep; the two friction rows of a point are consecutive: one load per pair when B is even
                if ((B & 1) != 0 || (k & 1) == 0) tot = sLam[NL + ((pos0 + k) >> 1)];
                const bool on = tot > 0.f;
                hi[k] = on ? mu * tot : lam[k]; lo[k] = on ? -hi[k] : lam[k];   // normal impulse not positive: the row is skipped
            } else { lo[k] = 0.f; hi[k] = (SEC == kSecLimit) ? 100.f : 1e10f; }     // joint limits [0, 100], contact normals [0, inf)
        }
        {
            int o = 0;
#pragma unroll
            for (int k = 1; k < B; ++k)
#pragma unroll
                for (int j = 0; j < k; ++j) ain[o++] = a_pair(ik[k], ik[j], tk[k], tk[j]);
        }
#pragma unroll
        for (int s = 0; s < S; ++s)
#pragma unroll
            for (int k = 0; k < B; ++k) ao[s][k] = a_own(s, ik[k], tk[k]);
#pragma unroll
        for (int k = 0; k < B; ++k) {
            float sel = w[0];
#pragma unroll
            for (int s = 1; s < S; ++s) if (ik[k] >= s * W) sel = w[s];
            wk[k] = T::shfl(sel, (S == 1) ? ik[k] : (ik[k] & (W - 1)));   // one row per lane: the row index is the owner's lane (the shuffle wraps indices past W itself)
        }
#pragma unroll
        for (int k = 0; k < B; ++k) {
            float c = fmaxf(fmaf(-inv[k], wk[k], rhs[k]), lo[k] - lam[k]);
            if (SEC != kSecNormal) c = fminf(c, hi[k] - lam[k]);     // contact normals have no upper bound (Bullet: 1e10)
            c = vk[k] ? c : 0.f;
#pragma unroll
            for (int j = k + 1; j < B; ++j) wk[j] = fmaf(ain[j * (j - 1) / 2 + k], c, wk[j]);
            if (vk[k] && writer[k]) sLam[ik[k]] = (SEC == kSecNormal) ? fmaxf(lam[k] + c, 0.f) : fminf(fmaxf(lam[k] + c, lo[k]), hi[k]);
#pragma unroll
            for (int s = 0; s < S; ++s) w[s] = fmaf(ao[s][k], c, w[s]);
        }
        __syncwarp();
    };
#pragma unroll 1
    for (int it = 0; it < 10; ++it) {
#pragma unroll 1
        for (int p0 = 0; p0 < NLmax; p0 += B) block(p0, it, std::integral_constant<int, kSecLimit>{});
#pragma unroll 1
        for (int p0 = 0; p0 < Pmax; p0 += B) block(p0, it, std::integral_constant<int, kSecNormal>{});
#pragma unroll 1
        for (int p0 = 0; p0 < 2 * Pmax; p0 += B) block(p0, it, std::integral_constant<int, kSecFriction>{});
    }
}

// Constraint rows of one Bullet sub-step for the environment owned by this tile (warp-collective; both environments of a W = 16 warp
// run it in lockstep).  Input (shared memory): per-link factors U / 1/D, joint axes, pivots, link velocities, contact points, limit
// rows, base Cholesky factor.  Output: impulses in sLam (also written to the persistent manifold), z = Y^T lambda in sZ.
// Row ids in solver order: limits [0,NL) | normals [NL, NL+P) | friction pairs NL+P+2p+{0,1} (t1 = -x, t2 = +z).
template <int W>
__device__ __noinline__ void solve_rows(int NL, int P, float* mani, int alive, unsigned int* prf) {
    using T = Tl<W>;
    // context from threadIdx and the block-shared header (nothing but scalars crosses the call, see Ctx below)
    float* const sm_ = step_smem();
    const int* LYS = reinterpret_cast<const int*>(sm_ + kHLayout);
    const float* LK = sm_ + kHdrFloats;
    const int lane = threadIdx.x % W;
    const float h = sm_[kHh], mu = sm_[kHMu];
#ifdef DM_PROFILE
    unsigned int pt = static_cast<unsigned int>(clock64());
#define SPROF(sec) do { if ((threadIdx.x & 31) == 0) { unsigned int t_ = static_cast<unsigned int>(clock64()); prf[sec] += t_ - pt; pt = t_; } } while (0)
#else
#define SPROF(sec) do { } while (0)
#endif
    const StepLayout& LY = *reinterpret_cast<const StepLayout*>(LYS);
    const int nl = LY.nl, CL = LY.chain_len, MR = LY.maxrows;
    constexpr int YS = dm_step_y_stride(W);   // row stride of Yt (>= maxrows: the host caps the row capacity there)
    float* const E = sm_ + LY.hot_floats + (threadIdx.x / W) * LY.env_floats;
    const unsigned char* CD = reinterpret_cast<const unsigned char*>(LK + nl * kLkFloats);
    const unsigned char* CH = CD + nl * nl;
    float* sU = E + LY.oU; float* sS = E + LY.oR; float* sW = E + LY.oW; float* sV = E + LY.oV; float* sA = E + LY.oA; float* sY = E + LY.oY;
    float* sLam = E + LY.oLam; float2* sRI = reinterpret_cast<float2*>(E + LY.oRhs); int* sRl = reinterpret_cast<int*>(E + LY.oRl);
    float* sPp = E + LY.oPp; float* sPi = E + LY.oPi; int* sPr = reinterpret_cast<int*>(E + LY.oPr);
    float* sQ = E + LY.oQ; float* sG = E + LY.oG; float* sZ = E + LY.oZ;
    auto lk_i = [&](int j) { return reinterpret_cast<const int*>(LK + j * kLkFloats)[kLInt]; };
    auto lk_i2 = [&](int j) { return reinterpret_cast<const int*>(LK + j * kLkFloats)[kLInt2]; };
    auto shift_f = [](S6 f, V3 c) { return mks(f.a + cross(c, f.l), f.l); };
    const int NR = NL + 3 * P;
    const int NRmax = (W == 32) ? NR : wmax(NR);
    const int nslots = (NRmax + W - 1) / W;
    constexpr int kPgsBlock = 2;   // solver steps evaluated per block of the projected Gauss-Seidel sweeps (measured on a B200: 1 -> 1.22 M, 2 -> 1.49 M, 4 -> 1.32 M, 8 -> 0.95 M policy steps/s)
    constexpr int kSlots = 2;   // rows per lane in the general path: the host caps the row capacity at dm_step_y_stride(W) (32 humanoid3d, 52 dog3d)
#pragma unroll
    for (int s = 0; s < kSlots; ++s) {
        const int rid = lane + s * W;
        if (s < nslots) {
            const bool rv_ = rid < NR;
            int b = 0, kind = 0 /*0 limit 1 normal 2 t1 3 t2*/, p = 0;
            float lsign = 1.f, lpen = 0.f;
            if (rv_) {
                if (rid < NL) { b = __float_as_int(sQ[rid]); lsign = sQ[8 + rid]; lpen = sQ[16 + rid]; }
                else if (rid < NL + P) { kind = 1; p = rid - NL; b = sPr[p] >> 2; }
                else { const int f = rid - NL - P; p = f >> 1; kind = 2 + (f & 1); b = sPr[p] >> 2; }
                sRl[rid] = b;
            }
            // unit force of the row on link b, about b's pivot, world axes
            S6 f = mks(mk3(0, 0, 0), mk3(0, 0, 0));
            float rvel = 0.f, pdist = 0.f;
            if (rv_ && kind != 0) {
                const float* w = sW + b * 12;
                pdist = sPp[p * 4 + 3];
                const V3 rel = mk3(sPp[p * 4] - w[9], sPp[p * 4 + 1] - w[10], sPp[p * 4 + 2] - w[11]);
                const V3 fl_ = (kind == 1) ? mk3(0.f, 1.f, 0.f) : ((kind == 2) ? mk3(-1.f, 0.f, 0.f) : mk3(0.f, 0.f, 1.f));
                f = mks(cross(rel, fl_), fl_);
                const float* v = sV + b * 12;
                rvel = dot(fl_, mk3(v[3], v[4], v[5]) + cross(mk3(v[0], v[1], v[2]), rel));
            }
            // walk the chain base <- ... <- b
            float acc = 0.f;
            int cur = b;
            bool first = true;
#pragma unroll 1
            while (true) {
                const int info = lk_i(cur);
                const int par = static_cast<int>(static_cast<signed char>(info & 0xff)), nd = (info >> 16) & 0xff, dp0 = (info >> 24) & 0xff;
                const float4* u4 = reinterpret_cast<const float4*>(sU + cur * 24);
                const float4* q4 = reinterpret_cast<const float4*>(sS + cur * 12);
                const float4 ua = u4[0], ub = u4[1], uc = u4[2], ud = u4[3], ue = u4[4], uf = u4[5];   // U0 U1 U2 | 1/D | sqrt(1/D)
                const float4 qa = q4[0], qb = q4[1], qc = q4[2];                                        // S0 S1 S2 | cw
                if (nd == 3) {
                    {   // dof 2
                        const float t = qb.z * f.a.x + qb.w * f.a.y + qc.x * f.a.z;
                        const float y = t * uf.w;
                        if (rv_) sY[(dp0 + 2) * YS + rid] = y;
                        acc += y * y;
                        const float ti = t * uf.x;
                        f.a.x -= ti * ud.x; f.a.y -= ti * ud.y; f.a.z -= ti * ud.z; f.l.x -= ti * ud.w; f.l.y -= ti * ue.x; f.l.z -= ti * ue.y;
                    }
                    {   // dof 1
                        const float t = qa.w * f.a.x + qb.x * f.a.y + qb.y * f.a.z;
                        const float y = t * uf.z;
                        if (rv_) sY[(dp0 + 1) * YS + rid] = y;
                        acc += y * y;
                        const float ti = t * ue.w;
                        f.a.x -= ti * ub.z; f.a.y -= ti * ub.w; f.a.z -= ti * uc.x; f.l.x -= ti * uc.y; f.l.y -= ti * uc.z; f.l.z -= ti * uc.w;
                    }
                }
                if (nd >= 1) {   // dof 0
                    float t = qa.x * f.a.x + qa.y * f.a.y + qa.z * f.a.z;
                    if (first && kind == 0) { t = lsign; rvel = lsign * sQ[24 + rid]; }
                    const float y = t * uf.y;
                    if (rv_) sY[dp0 * YS + rid] = y;
                    acc += y * y;
                    const float ti = t * ue.z;
                    f.a.x -= ti * ua.x; f.a.y -= ti * ua.y; f.a.z -= ti * ua.z; f.l.x -= ti * ua.w; f.l.y -= ti * ub.x; f.l.z -= ti * ub.y;
                }
                first = false;
                f = shift_f(f, mk3(qc.y, qc.z, qc.w));
                if (par < 0) break;
                cur = par;
            }
            {   // base block: y = G^-1 f
                float x[6] = {f.a.x, f.a.y, f.a.z, f.l.x, f.l.y, f.l.z};
                int o = 0;
#pragma unroll
                for (int i = 0; i < 6; ++i) {
#pragma unroll
                    for (int k = 0; k < i; ++k) x[i] -= sG[o++] * x[k];
                    x[i] *= sG[15 + i];
                    if (rv_) sY[i * YS + rid] = x[i];
                    acc += x[i] * x[i];
                }
            }
            if (rv_) {
                const float inv = acc > 1.1920929e-7f ? 1.0f / acc : 0.f;
                float rhs, lam0 = 0.f;
                if (kind == 1) {   // setupMultiBodyContactConstraint: erp 0.2, restitution 0, no split impulse for multibodies
                    float perr = 0.f, verr = -rvel;
                    if (pdist > 0.f) verr -= pdist / h; else perr = -pdist * 0.2f / h;
                    rhs = perr * inv + verr * inv;
                    lam0 = sPi[p] * 0.85f;   // SOLVER_USE_WARMSTARTING, warmstartingFactor 0.85
                } else if (kind != 0) rhs = -rvel * inv;
                else {
                    float perr = 0.f, verr = -rvel;
                    const bool combine = lpen > -0.04f;   // split-impulse threshold: deeper violations lose the positional term (btMultiBodyJointLimitConstraint)
                    if (lpen > 0.f) verr = -lpen / h; else perr = -lpen * 0.2f / h;
                    rhs = combine ? (perr * inv + verr * inv) : (verr * inv);
                }
                sRI[rid] = make_float2(rhs, inv); sLam[rid] = lam0;
            }
        }
    }
    __syncwarp();
    SPROF(7);
    const int Pmax = (W == 32) ? P : wmax(P);
    const int NLmax = (W == 32) ? NL : wmax(NL);
    {
        // ---- A = J M^-1 J^T = Y Y^T: lanes = (i, j <= i) pairs of the lower triangle, W pairs per pass.  At most W rows (the common case): full
        // symmetric W x W square (stride W); more: packed lower triangle (pair index = storage index).  Overwrites the world-frame / velocity
        // scratch, no longer needed this sub-step.
        // storage: 0 = W x W square (one row per lane), 1 = kSq2 x kSq2 square on two rows per lane (most "more than W rows" cases are just above
        // W; its sweep blocks are ~75 instructions against ~95 with packed indexing), 2 = packed triangle (pair index = storage index).
        // Warp-uniform (NRmax).
        constexpr int kSq2 = (W == 16) ? 22 : 36;             // kSq2^2 floats fit the scratch block (dm_step_layout: max(24 nl, maxrows (maxrows + 1) / 2))
        const int region = max(nl * 24, MR * (MR + 1) / 2);   // floats of the scratch block
        const int mode = (nslots == 1) ? 0 : ((NRmax <= kSq2 && kSq2 * kSq2 + W <= region) ? 1 : 2);
        const int st = (mode == 0) ? W : kSq2;
        auto put = [&](int i, int j, float v) {   // A(i, j) = A(j, i) = v
            if (mode != 2) { sA[i * st + j] = v; sA[j * st + i] = v; }
            else { const int hi_ = max(i, j), lo_ = min(i, j); sA[hi_ * (hi_ + 1) / 2 + lo_] = v; }
        };
        // (1) pairs with a joint-limit row (rows [0, NL): the smaller index of such a pair is a limit row): lanes = the other row
#pragma unroll 1
        for (int j = 0; j < NLmax; ++j) {
            const bool jv = j < NL;
            const int bj = jv ? sRl[j] : 0;
#pragma unroll 1
            for (int i0 = 0; i0 < NRmax; i0 += W) {
                const int i = i0 + lane;
                const bool pv = jv && i < NR && i >= j;
                const int cd = pv ? CD[sRl[i] * nl + bj] : 0;          // common chain depth of rows i and j
                const float* yi = sY + (pv ? i : 0); const float* yj = sY + (jv ? j : 0);
                float acc = 0.f;
#pragma unroll 1
                for (int k = 0; k < CL; k += 4, yi += 4 * YS, yj += 4 * YS) {   // entries past the common depth are masked (reads past the chain length stay inside the block)
                    const float a0 = yi[0], a1 = yi[YS], a2 = yi[2 * YS], a3 = yi[3 * YS];
                    const float b0 = yj[0], b1 = yj[YS], b2 = yj[2 * YS], b3 = yj[3 * YS];
                    if (k < cd) acc += a0 * b0;
                    if (k + 1 < cd) acc += a1 * b1;
                    if (k + 2 < cd) acc += a2 * b2;
                    if (k + 3 < cd) acc += a3 * b3;
                }
                if (pv) put(i, j, acc);
            }
        }
        // (2) contact rows: lanes = (p, r <= p) pairs of contact POINTS, each lane forms the 3 x 3 block between the rows {normal, t1, t2} of the
        // two points (rows NL + p, NL + P + 2 p, NL + P + 2 p + 1: they act on the same link, so one common depth serves all nine products, and
        // six Y rows are loaded for nine dot products instead of two per product).  Same products, same summation order as pair by pair.
        const int npp = P * (P + 1) / 2, nppmax = Pmax * (Pmax + 1) / 2;
#pragma unroll 1
        for (int q0 = 0; q0 < nppmax; q0 += W) {
            const int q = q0 + lane;
            const bool pv = q < npp;
            int pp = static_cast<int>((sqrtf(8.0f * static_cast<float>(q) + 1.0f) - 1.0f) * 0.5f);
            if (pp * (pp + 1) / 2 > q) --pp;
            if ((pp + 1) * (pp + 2) / 2 <= q) ++pp;
            const int pr = q - pp * (pp + 1) / 2;
            const int in_p = pv ? NL + pp : 0, it_p = pv ? NL + P + 2 * pp : 0, in_r = pv ? NL + pr : 0, it_r = pv ? NL + P + 2 * pr : 0;
            const int cd = pv ? CD[sRl[in_p] * nl + sRl[in_r]] : 0;
            const float* ypn = sY + in_p; const float* ypt = sY + it_p; const float* yrn = sY + in_r; const float* yrt = sY + it_r;
            float acc[3][3];
#pragma unroll
            for (int x = 0; x < 3; ++x)
#pragma unroll
                for (int y = 0; y < 3; ++y) acc[x][y] = 0.f;
#pragma unroll 1
            for (int k = 0; k < CL; k += 4, ypn += 4 * YS, ypt += 4 * YS, yrn += 4 * YS, yrt += 4 * YS) {
                float av[3][4], bv[3][4];
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    av[0][d] = ypn[d * YS]; av[1][d] = ypt[d * YS]; av[2][d] = ypt[d * YS + 1];
                    bv[0][d] = yrn[d * YS]; bv[1][d] = yrt[d * YS]; bv[2][d] = yrt[d * YS + 1];
                }
#pragma unroll
                for (int d = 0; d < 4; ++d)
                    if (k + d < cd) {
#pragma unroll
                        for (int x = 0; x < 3; ++x)
#pragma unroll
                            for (int y = 0; y < 3; ++y) acc[x][y] += av[x][d] * bv[y][d];
                    }
            }
            if (pv) {
                if (mode != 2) {   // square: rows of p at stride st, columns of r, and the transposed entries
                    float* rp[3] = {sA + in_p * st, sA + it_p * st, sA + it_p * st + st};
                    float* rr[3] = {sA + in_r * st, sA + it_r * st, sA + it_r * st + st};
                    const int cp[3] = {in_p, it_p, it_p + 1}, cr[3] = {in_r, it_r, it_r + 1};
#pragma unroll
                    for (int x = 0; x < 3; ++x)
#pragma unroll
                        for (int y = 0; y < 3; ++y) { rp[x][cr[y]] = acc[x][y]; rr[y][cp[x]] = acc[x][y]; }
                } else {
#pragma unroll
                    for (int x = 0; x < 3; ++x)
#pragma unroll
                        for (int y = 0; y < 3; ++y) put(x == 0 ? in_p : it_p + x - 1, y == 0 ? in_r : it_r + y - 1, acc[x][y]);
                }
            }
        }
        __syncwarp();
        SPROF(8);
        if (mode == 0) pgs_sweeps<W, 1, W, kPgsBlock>(sA, sLam, sRI, lane, NL, P, NLmax, Pmax, mu);
        else if (mode == 1) pgs_sweeps<W, kSlots, kSq2, kPgsBlock>(sA, sLam, sRI, lane, NL, P, NLmax, Pmax, mu);
        else pgs_sweeps<W, kSlots, 0, kPgsBlock>(sA, sLam, sRI, lane, NL, P, NLmax, Pmax, mu);
    }
    SPROF(9);
    // write impulses back to the manifold (warm start of the next sub-step)
#pragma unroll 1
    for (int p = lane; p < P; p += W) {
        if (alive) {
            const int ref = sPr[p];
            float* mpt = mani + (ref >> 2) * kManifoldFloats + (ref & 3) * 12;
            mpt[7] = sLam[NL + p]; mpt[8] = sLam[NL + P + 2 * p]; mpt[9] = sLam[NL + P + 2 * p + 1];
        }
    }
    // ---- z = Y^T lambda: lane = link accumulates the entries of its own dofs over the rows whose chain passes through it; lanes < 6 also
    // accumulate the base entry of the same index
    {
        const int info = (lane < nl) ? lk_i(lane) : 0;
        const int nd = (info >> 16) & 0xff, dp0 = (info >> 24) & 0xff;
        const int d0 = (lane < nl) ? (lk_i2(lane) & 0xff) : 0;
        float z0 = 0.f, z1 = 0.f, z2 = 0.f, zb = 0.f;
        const int kb = (lane < 6) ? lane : 0;
        // branch-free body, loads independent of the accumulators (two rows in flight): rows past NR contribute lambda = 0 (their Y entries are
        // initialised words of the block), links outside the row's chain are masked
        const bool mine = lane < nl && nd > 0;
        const int need = dp0 + nd - 1;
        const unsigned char* cdl = CD + lane;
#pragma unroll 2
        for (int i = 0; i < NRmax; ++i) {
            const int b = sRl[i];
            const float l = (i < NR) ? sLam[i] : 0.f;
            const float yb = sY[kb * YS + i], y0 = sY[dp0 * YS + i], y1 = sY[(dp0 + 1) * YS + i], y2 = sY[(dp0 + 2) * YS + i];
            const bool in = mine && cdl[b * nl] > need;   // the row's chain contains this link's dofs
            zb = fmaf(yb, l, zb);
            if (in) { z0 = fmaf(y0, l, z0); if (nd == 3) { z1 = fmaf(y1, l, z1); z2 = fmaf(y2, l, z2); } }
        }
        if (lane < 6) sZ[lane] = zb;
        if (lane < nl && nd >= 1) sZ[d0] = z0;
        if (lane < nl && nd == 3) { sZ[d0 + 1] = z1; sZ[d0 + 2] = z2; }
    }
    __syncwarp();
}


// ---- per-lane context of the phase routines.  The routines are real calls (__noinline__: each gets the whole register budget), and a struct
// passed by value to a real call travels through the caller's local-memory stack: every field access in the callee was a local load (the
// ncu capture of round 2 showed 28 % of the stall samples on those).  So nothing is passed: a routine rebuilds its context from threadIdx and
// the block-shared tables (two LDS), and the launch constants (layout, gravity, h, ...) sit in a header in front of the link table.
struct Ctx {
    float* E;              // this environment's shared-memory block
    const int* LYS;        // layout (shared copy of StepLayout)
    const float* LK;       // block-shared link constants
    int lane, li;          // lane in the tile, link index (clamped for idle lanes)
    int plane, level, ndof, jtype, maxlevel;   // kinematic tree (the articulated-body passes read their dynamics tree themselves)
    bool act;
};
__device__ __forceinline__ const StepLayout& lay_of(const Ctx& c) { return *reinterpret_cast<const StepLayout*>(c.LYS); }
template <int W>
__device__ __forceinline__ Ctx make_ctx() {
    Ctx c;
    float* sm = step_smem();
    c.LYS = reinterpret_cast<const int*>(sm + kHLayout); c.LK = sm + kHdrFloats;
    const StepLayout& LY = *reinterpret_cast<const StepLayout*>(c.LYS);
    const int tile = threadIdx.x / W;
    c.lane = threadIdx.x % W;
    c.act = c.lane < LY.nl;
    c.li = c.act ? c.lane : LY.nl - 1;
    c.E = sm + LY.hot_floats + tile * LY.env_floats;
    const int* q = reinterpret_cast<const int*>(c.LK + c.li * kLkFloats);
    const int info = q[kLInt], tree = q[kLTree];
    const int par = static_cast<int>(static_cast<signed char>(info & 0xff));
    c.plane = par >= 0 ? par : 0; c.jtype = (info >> 8) & 0xff; c.ndof = c.act ? ((info >> 16) & 0xff) : 0;
    c.level = c.act ? (tree & 0xff) : 1000; c.maxlevel = (tree >> 8) & 0xff;
    return c;
}
__device__ __forceinline__ S6 shift_m(S6 m, V3 c) { return mks(m.a, m.l + cross(m.a, c)); }   // motion vector: reference point moved by +c
__device__ __forceinline__ S6 shift_f(S6 f, V3 c) { return mks(f.a + cross(c, f.l), f.l); }   // force vector: child pivot -> parent pivot (child = parent + c)
__device__ __forceinline__ float cl100(float v) { return fminf(fmaxf(v, -100.f), 100.f); }   // applyDeltaVeeMultiDof clamp
// cSimCharacter::CalcCOM (SimCharacter.cpp:398-416) over the lanes of one environment: w = this link's sW entry (pivot at [9..11]),
// v = its sV entry (pivot -> COM at [6..8]), both as left by kin_pass; returns the unscaled COM on every lane of the tile
template <int W>
__device__ __forceinline__ V3 tile_com(const float* w, const float* v, float mass, float inv_total) {
    float cx = mass * (w[9] + v[6]), cy = mass * (w[10] + v[7]), cz = mass * (w[11] + v[8]);
#pragma unroll
    for (int o = W / 2; o > 0; o >>= 1) {
        cx += __shfl_xor_sync(0xffffffffu, cx, o, W); cy += __shfl_xor_sync(0xffffffffu, cy, o, W); cz += __shfl_xor_sync(0xffffffffu, cz, o, W);
    }
    return mk3(cx * inv_total, cy * inv_total, cz * inv_total);
}

// Forward kinematics and link velocities, root -> leaves.  Writes per link: world->link rotation + pivot (sW), joint axes in world axes +
// parent pivot -> pivot (sS), spatial velocity at the pivot + pivot -> COM (sV).  Base state is read from sB by lane 0.
template <int W>
__device__ __noinline__ void kin_pass(float4 jp, float4 jv) {
    const Ctx c = make_ctx<W>();
    using T = Tl<W>;
    const StepLayout& LY = lay_of(c);
    float* sS = c.E + LY.oR; float* sW = c.E + LY.oW; float* sV = c.E + LY.oV; const float* sB = c.E + LY.oG + 21;
    const float* LKo = c.LK + c.li * kLkFloats;
    const float4 ax4 = ld4(LKo + kLAx), zr4 = ld4(LKo + kLZr), c4 = ld4(LKo + kLC);
    const V3 axis = mk3(ax4.x, ax4.y, ax4.z);
    const Q4 zrot = mkq(zr4.x, zr4.y, zr4.z, zr4.w);
    const V3 cvec = mk3(c4.x, c4.y, c4.z);
    Q4 cached;
    if (c.jtype == kJSpherical) cached = qmul(mkq(jp.x, jp.y, jp.z, -jp.w), zrot);
    else if (c.jtype == kJRevolute) {
        float s, co;
        __sincosf(-0.5f * jp.x, &s, &co);   // |angle| <= pi/2 + limit overshoot: fast path is accurate to ~1 ulp of the result scale
        cached = qmul(mkq(axis.x * s, axis.y * s, axis.z * s, co), zrot);
    } else cached = zrot;
    const M3 R = qmat(cached);
    V3 jw = mk3(0, 0, 0);
    if (c.jtype == kJSpherical) jw = mk3(jv.x, jv.y, jv.z); else if (c.jtype == kJRevolute) jw = jv.x * axis;
    M3 Rwl; V3 Pw, cw; S6 vel;
    if (c.lane == 0) {
        const M3 Rwb = qmat(mkq(sB[3], sB[4], sB[5], sB[6]));
        const V3 bo = mk3(sB[7], sB[8], sB[9]);
        Rwl = mul(R, Rwb); cw = mulT(Rwb, cvec); Pw = mk3(sB[0], sB[1], sB[2]) + cw;
        vel = mks(bo + mulT(Rwl, jw), mk3(sB[10], sB[11], sB[12]) + cross(bo, cw));
    }
#pragma unroll 1
    for (int lv = 1; lv <= c.maxlevel; ++lv) {
        M3 pR; V3 pp; S6 pv;
#pragma unroll
        for (int k = 0; k < 9; ++k) pR.m[k] = T::shfl(Rwl.m[k], c.plane);
        pp = T::shfl3(Pw, c.plane);
        pv = T::shfl6(vel, c.plane);
        if (c.level == lv) {
            Rwl = mul(R, pR); cw = mulT(pR, cvec); Pw = pp + cw;
            vel = mks(pv.a + mulT(Rwl, jw), pv.l + cross(pv.a, cw));
        }
    }
    if (c.act) {
        const float4 d4 = ld4(LKo + kLD);
        const V3 dw = mulT(Rwl, mk3(d4.x, d4.y, d4.z));
        V3 S0 = mk3(Rwl.m[0], Rwl.m[1], Rwl.m[2]);
        if (c.jtype != kJSpherical) S0 = mulT(Rwl, axis);
        const float wr[12] = {Rwl.m[0], Rwl.m[1], Rwl.m[2], Rwl.m[3], Rwl.m[4], Rwl.m[5], Rwl.m[6], Rwl.m[7], Rwl.m[8], Pw.x, Pw.y, Pw.z};
        const float qr[12] = {S0.x, S0.y, S0.z, Rwl.m[3], Rwl.m[4], Rwl.m[5], Rwl.m[6], Rwl.m[7], Rwl.m[8], cw.x, cw.y, cw.z};
        const float vr[12] = {vel.a.x, vel.a.y, vel.a.z, vel.l.x, vel.l.y, vel.l.z, dw.x, dw.y, dw.z, 0.f, 0.f, 0.f};
        st12(sW + c.lane * 12, wr); st12(sS + c.lane * 12, qr); st12(sV + c.lane * 12, vr);
    }
    __syncwarp();
}

// Collision of this lane's link with the plane y = 0: persistent manifold of <= 4 points (btPersistentManifold), one new point per
// sub-step from the support vertex (btConvexPlaneCollisionAlgorithm), refresh with the breaking threshold.  The manifold lives in global
// memory; the points of the environment are published to shared memory for the row builder.
// Returns P | in_contact_tol << 8 | overflow << 9 | this lane's point count << 10.
template <int W>
__device__ __noinline__ int collide(float* mani, int alive, int mcnt) {
    const Ctx c = make_ctx<W>();
    const float scale = step_smem()[kHScale];
    using T = Tl<W>;
    const StepLayout& LY = lay_of(c);
    const float* sW = c.E + LY.oW; const float* sV = c.E + LY.oV;
    float* sPp = c.E + LY.oPp; float* sPi = c.E + LY.oPi; int* sPr = reinterpret_cast<int*>(c.E + LY.oPr);
    const float* LKo = c.LK + c.li * kLkFloats;
    const int shape = reinterpret_cast<const int*>(LKo)[kLFlg] & 0xff;
    int cnt = 0;
    float mp[48];
    M3 Rwl;
    float wrec[12], vrec[12];
    ld12(sW + c.li * 12, wrec); ld12(sV + c.li * 12, vrec);
#pragma unroll
    for (int k = 0; k < 9; ++k) Rwl.m[k] = wrec[k];
    const float thr = LKo[kLThr];
    const float4 he4 = ld4(LKo + kLHe);
    const V3 he = mk3(he4.x, he4.y, he4.z);
    const V3 pos = mk3(wrec[9] + vrec[6], wrec[10] + vrec[7], wrec[11] + vrec[8]);   // COM, world (Bullet's link collider frame)
    V3 dl = mul(Rwl, mk3(0.f, -1.f, 0.f));   // support direction -n in link coordinates
    V3 vtx;
    if (shape == kSBox) vtx = mk3(dl.x >= 0 ? he.x : -he.x, dl.y >= 0 ? he.y : -he.y, dl.z >= 0 ? he.z : -he.z);
    else {
        V3 sup = mk3(0, 0, 0);
        if (shape == kSCapsule) sup = mk3(0.f, (dl.y >= 0.f) ? he.y : -he.y, 0.f);   // first end point wins ties
        float inv = rsqrtf(dot(dl, dl));
        vtx = sup + (he.x * inv) * dl;
    }
    const V3 vw = pos + mulT(Rwl, vtx);
    const float dist = vw.y;
    // The manifold of a link is read (and written back) only if it can matter: the link held points after the previous sub-step (mcnt, carried
    // by the caller; "unknown" = 4 at the start of a launch) or its support vertex is inside the contact threshold now.  For all other links --
    // 13 of 15 for a standing humanoid -- the twelve 16-byte loads and stores per lane are predicated off: with the warps of a block in lockstep
    // they all arrive here together, and the unconditional version throttled the memory pipe (14.6 % of the stall samples in capture r02y).
    const bool need = c.act && alive && (mcnt > 0 || dist < thr);
    {
        const float4* mg = reinterpret_cast<const float4*>(mani + c.li * kManifoldFloats);
#pragma unroll
        for (int k = 0; k < 12; ++k) { float4 v = need ? mg[k] : make_float4(0.f, 0.f, 0.f, 0.f); mp[4 * k] = v.x; mp[4 * k + 1] = v.y; mp[4 * k + 2] = v.z; mp[4 * k + 3] = v.w; }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) if (mp[k * 12] != 0.f && cnt == k) cnt = k + 1;
    if (c.act && dist < thr) {
        float best = thr * thr; int nearest = -1;
#pragma unroll
        for (int k = 0; k < 4; ++k) if (k < cnt) {
            float dx = mp[k * 12 + 1] - vtx.x, dy = mp[k * 12 + 2] - vtx.y, dz = mp[k * 12 + 3] - vtx.z, dd = dx * dx + dy * dy + dz * dz;
            if (dd < best) { best = dd; nearest = k; }
        }
        int idx = nearest;
        float k7 = 0, k8 = 0, k9 = 0, k11 = 0;
        if (nearest >= 0) {
#pragma unroll
            for (int k = 0; k < 4; ++k) if (k == nearest) { k7 = mp[k * 12 + 7]; k8 = mp[k * 12 + 8]; k9 = mp[k * 12 + 9]; k11 = mp[k * 12 + 11]; }
        } else if (cnt < 4) { idx = cnt; cnt++; }
        else {   // btPersistentManifold::sortCachedPoints
            int mpi = -1; float mpen = dist;
#pragma unroll
            for (int k = 0; k < 4; ++k) if (mp[k * 12 + 10] < mpen) { mpi = k; mpen = mp[k * 12 + 10]; }
            auto Pt = [&](int k) { return mk3(mp[k * 12 + 1], mp[k * 12 + 2], mp[k * 12 + 3]); };
            auto area = [&](V3 a, V3 b) { V3 x = cross(a, b); return dot(x, x); };
            float res[4] = {0, 0, 0, 0};
            if (mpi != 0) res[0] = area(vtx - Pt(1), Pt(3) - Pt(2));
            if (mpi != 1) res[1] = area(vtx - Pt(0), Pt(3) - Pt(2));
            if (mpi != 2) res[2] = area(vtx - Pt(0), Pt(3) - Pt(1));
            if (mpi != 3) res[3] = area(vtx - Pt(0), Pt(2) - Pt(1));
            idx = 0; float bv = fabsf(res[0]);
#pragma unroll
            for (int k = 1; k < 4; ++k) if (fabsf(res[k]) > bv) { bv = fabsf(res[k]); idx = k; }
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) if (k == idx) {
            float* q = mp + k * 12;
            q[0] = 1.f; q[1] = vtx.x; q[2] = vtx.y; q[3] = vtx.z; q[4] = vw.x; q[5] = 0.f; q[6] = vw.z; q[7] = k7; q[8] = k8; q[9] = k9; q[10] = dist; q[11] = k11;
        }
    }
    // refreshContactPoints
#pragma unroll
    for (int k = 3; k >= 0; --k) if (k < cnt) {
        V3 pa = pos + mulT(Rwl, mk3(mp[k * 12 + 1], mp[k * 12 + 2], mp[k * 12 + 3]));
        mp[k * 12 + 10] = pa.y - mp[k * 12 + 5];
        mp[k * 12 + 11] += 1.f;
    }
#pragma unroll
    for (int k = 3; k >= 0; --k) if (k < cnt) {
        V3 pa = pos + mulT(Rwl, mk3(mp[k * 12 + 1], mp[k * 12 + 2], mp[k * 12 + 3]));
        bool rm = !(mp[k * 12 + 10] <= thr);
        if (!rm) {
            float dx = mp[k * 12 + 4] - pa.x, dy = mp[k * 12 + 5] - (pa.y - mp[k * 12 + 10]), dz = mp[k * 12 + 6] - pa.z;
            rm = (dx * dx + dy * dy + dz * dz) > thr * thr;
        }
        if (rm) {
            const int last = cnt - 1;
#pragma unroll
            for (int l2 = 0; l2 < 4; ++l2) if (l2 == last) {
                if (k != l2) for (int j = 0; j < 12; ++j) mp[k * 12 + j] = mp[l2 * 12 + j];
                mp[l2 * 12] = 0.f;
            }
            cnt--;
        }
    }
    if (!c.act || !alive) cnt = 0;   // finished episodes are frozen until dm_reset: no constraint rows for them
    int tol = 0;                     // cContactManager::Update: distance <= 0.001 * scale
#pragma unroll
    for (int k = 0; k < 4; ++k) if (k < cnt && mp[k * 12 + 10] <= 0.001f * scale) tol = 1;
    if (need) {
        float4* mo = reinterpret_cast<float4*>(mani + c.li * kManifoldFloats);
#pragma unroll
        for (int k = 0; k < 12; ++k) mo[k] = make_float4(mp[4 * k], mp[4 * k + 1], mp[4 * k + 2], mp[4 * k + 3]);
    }
    // exclusive prefix over lanes -> point indices; publish points to the solver
    int incl = cnt, over = 0;
#pragma unroll
    for (int o = 1; o < W; o <<= 1) { int t = __shfl_up_sync(0xffffffffu, incl, o, W); if (c.lane >= o) incl += t; }
    const int base = incl - cnt;
#pragma unroll
    for (int k = 0; k < 4; ++k) if (k < cnt) {
        const int p = base + k;
        if (p < LY.maxpts) {
            V3 pa = pos + mulT(Rwl, mk3(mp[k * 12 + 1], mp[k * 12 + 2], mp[k * 12 + 3]));
            sPp[p * 4] = pa.x; sPp[p * 4 + 1] = pa.y; sPp[p * 4 + 2] = pa.z; sPp[p * 4 + 3] = mp[k * 12 + 10];
            sPi[p] = mp[k * 12 + 7];
            sPr[p] = c.lane * 4 + k;
        } else over = 1;
    }
    const int P = min(T::shfli(incl, W - 1), LY.maxpts);
    __syncwarp();
    return P | (tol << 8) | (over << 9) | (cnt << 10);
}

// Articulated-body solve of  H qdd = g - C  for this environment (H: joint-space inertia, + kdt on the joint diagonal for Stable-PD).
//   root -> leaves: bias accelerations; leaves -> root: articulated inertia IA and bias force pA, one scalar elimination per dof
//   (deepest first) = one step of the tree-structured L^T D L; base: 6x6 Cholesky in world axes (= the generalised base coordinates);
//   root -> leaves: accelerations.  Bullet sub-steps (bullet != 0) also publish the factors (sU, sG), advance the link velocities in sV
//   and the base velocity in sB by h * acceleration.  Returns this link's joint accelerations.
template <int W, bool DEBUG>
__device__ __noinline__ float3 aba_solve(float g0, float g1, float g2, float kdt, int bullet, float jvx, float jvy, float jvz, float* dbg_acc) {
    const Ctx c = make_ctx<W>();
    const float gx = step_smem()[kHGrav], gy = step_smem()[kHGrav + 1], gz = step_smem()[kHGrav + 2], h = step_smem()[kHh];
    using T = Tl<W>;
    const StepLayout& LY = lay_of(c);
    float* sU = c.E + LY.oU; const float* sS = c.E + LY.oR; const float* sW = c.E + LY.oW; float* sV = c.E + LY.oV; float* sG = c.E + LY.oG; float* sB = sG + 21;
    const float* LKo = c.LK + c.li * kLkFloats;
    // dynamics tree (see the table build in dm_step_kernel): parent lane, level (root -1: its lane accumulates the base; lumped fixed leaves 100:
    // they take no part), the bypassed root whose pivot offset is added to this link's shift, children
    const int dyn = c.act ? reinterpret_cast<const int*>(LKo)[kLDyn] : (100 << 8);
    const int dpar = dyn & 0xff, dlev = static_cast<int>(static_cast<signed char>((dyn >> 8) & 0xff)), byp = (dyn >> 16) & 0xff, dnch = (dyn >> 24) & 0xff;
    const int dchild = reinterpret_cast<const int*>(LKo)[kLDChild];
    const int dmax = reinterpret_cast<const int*>(step_smem())[kHDmax];
    const bool isroot = c.lane == 0;
    const float4 dc4 = ld4(LKo + kLDc);           // reference point -> composite COM (link axes) | composite mass
    const float mass = c.act ? dc4.w : 0.f;       // composite mass (own + lumped leaves; 0 for a lumped leaf itself)
    float q[12];
    ld12(sS + c.li * 12, q);
    const V3 S0 = mk3(q[0], q[1], q[2]), S1 = mk3(q[3], q[4], q[5]), S2 = mk3(q[6], q[7], q[8]), cwk = mk3(q[9], q[10], q[11]);   // cwk: kinematic parent's pivot -> pivot
    V3 cw = cwk;                                    // dynamics parent's reference point -> this link's reference point
    if (byp != 0xff) { const float* qb = sS + byp * 12; cw = cw + mk3(qb[9], qb[10], qb[11]); }
    if (isroot) cw = mk3(0, 0, 0);
    float vv[8];
    {
        const float4 a = reinterpret_cast<const float4*>(sV + c.li * 12)[0], b = reinterpret_cast<const float4*>(sV + c.li * 12)[1];
        vv[0] = a.x; vv[1] = a.y; vv[2] = a.z; vv[3] = a.w; vv[4] = b.x; vv[5] = b.y;
    }
    const S6 velk = mks(mk3(vv[0], vv[1], vv[2]), mk3(vv[3], vv[4], vv[5]));   // velocity at the link's own pivot
    S6 vel = velk;                                                               // velocity at the reference point of the dynamics (root: base origin)
    if (isroot) vel = mks(mk3(sB[7], sB[8], sB[9]), mk3(sB[10], sB[11], sB[12]));
    V3 jww = mk3(0, 0, 0);   // joint angular velocity, world axes
    if (c.jtype == kJSpherical) jww = jvx * S0 + jvy * S1 + jvz * S2; else if (c.jtype == kJRevolute) jww = jvx * S0;
    // ---- bias accelerations (root -> leaves)
    S6 ab;
    {
        const S6 cj = mks(cross(vel.a, jww), cross(vel.l, jww));
        if (isroot) {
            const V3 bo = vel.a, bv = vel.l;
            V3 wxv;
            if (bullet) wxv = cross(bo, bv);
            else {   // cRBDUtil::BuildCjRoot differentiates the root quaternion with the body-frame formula applied to the world-frame
                     // angular velocity (RBDUtil.cpp:915-958): reproduced in the Stable-PD stage
                const M3 Rwb = qmat(mkq(sB[3], sB[4], sB[5], sB[6]));
                wxv = mulT(Rwb, cross(bo, mul(Rwb, bv)));
            }
            ab = mks(mk3(0, 0, 0), mk3(-gx, -gy, -gz) - wxv);   // at the base origin (the root link has no joint velocity: no cj)
        }
#pragma unroll 1
        for (int lv = 0; lv <= dmax; ++lv) {
            S6 pa = T::shfl6(ab, dpar);
            if (dlev == lv) ab = shift_m(pa, cw) + cj;
        }
    }
    // ---- leaves -> root
    Art IA; S6 pA;
    float inv0 = 0.f, inv1 = 0.f, inv2 = 0.f, u0 = 0.f, u1 = 0.f, u2 = 0.f;
    {
        const float* wsel = LKo + (bullet ? kLWb : kLWd);
        const float4 w4 = ld4(wsel); const float2 w2 = *reinterpret_cast<const float2*>(wsel + 4);
        float wl[6] = {w4.x, w4.y, w4.z, w4.w, w2.x, w2.y};
#pragma unroll
        for (int k = 0; k < 6; ++k) wl[k] = c.act ? wl[k] : 0.f;
        M3 Rwl;
        {
            float w[12];
            ld12(sW + c.li * 12, w);
#pragma unroll
            for (int k = 0; k < 9; ++k) Rwl.m[k] = w[k];
        }
        rot_sym(Rwl, wl, IA.ww);     // link axes -> world axes
        const V3 md = mass * mulT(Rwl, mk3(dc4.x, dc4.y, dc4.z));   // first moment about the reference point, world axes
        IA.wv[0] = 0.f; IA.wv[1] = -md.z; IA.wv[2] = md.y; IA.wv[3] = md.z; IA.wv[4] = 0.f; IA.wv[5] = -md.x; IA.wv[6] = -md.y; IA.wv[7] = md.x; IA.wv[8] = 0.f;
        IA.vv[0] = mass; IA.vv[1] = 0.f; IA.vv[2] = 0.f; IA.vv[3] = mass; IA.vv[4] = 0.f; IA.vv[5] = mass;
        // h = I v ; pA = I ab + v x* h
        const V3 hn = sym_mul(IA.ww, vel.a) + cross(md, vel.l), hf = mass * vel.l + cross(vel.a, md);
        const V3 an = sym_mul(IA.ww, ab.a) + cross(md, ab.l), af = mass * ab.l + cross(ab.a, md);
        pA = mks(an + cross(vel.a, hn) + cross(vel.l, hf), af + cross(vel.a, hf));
    }
    // U_d = IA s_d goes straight to the environment's factor table (sU: read back by the acceleration pass below and, in the Bullet sub-steps,
    // by the constraint rows and the velocity correction) instead of living in 18 registers across the leaves -> root loop
    float* const uown = sU + c.lane * 24;
    float* const scr = c.E + LY.oY;   // 28 floats per lane (dm_step_layout guarantees the room and the 16-byte alignment)
    auto eliminate = [&](V3 dir, float g, int d, float& invo, float& uo) {
        const V3 Ua = sym_mul(IA.ww, dir), Ul = wvT_mul(IA.wv, dir);
        const float D = dot(dir, Ua) + kdt;
        const float inv = rcp_fast(D);   // MUFU.RCP (1 ulp); D = s . IA s + kdt is a positive, well-scaled inertia
        const float u = g - dot(dir, pA.a);
        const V3 sa = inv * Ua, sl = inv * Ul;
        IA.ww[0] -= sa.x * Ua.x; IA.ww[1] -= sa.x * Ua.y; IA.ww[2] -= sa.x * Ua.z; IA.ww[3] -= sa.y * Ua.y; IA.ww[4] -= sa.y * Ua.z; IA.ww[5] -= sa.z * Ua.z;
        IA.wv[0] -= sa.x * Ul.x; IA.wv[1] -= sa.x * Ul.y; IA.wv[2] -= sa.x * Ul.z; IA.wv[3] -= sa.y * Ul.x; IA.wv[4] -= sa.y * Ul.y; IA.wv[5] -= sa.y * Ul.z;
        IA.wv[6] -= sa.z * Ul.x; IA.wv[7] -= sa.z * Ul.y; IA.wv[8] -= sa.z * Ul.z;
        IA.vv[0] -= sl.x * Ul.x; IA.vv[1] -= sl.x * Ul.y; IA.vv[2] -= sl.x * Ul.z; IA.vv[3] -= sl.y * Ul.y; IA.vv[4] -= sl.y * Ul.z; IA.vv[5] -= sl.z * Ul.z;
        pA.a += u * sa; pA.l += u * sl;
        float2* uo_ = reinterpret_cast<float2*>(uown + 6 * d);   // 8-byte aligned: 24-float records
        uo_[0] = make_float2(Ua.x, Ua.y); uo_[1] = make_float2(Ua.z, Ul.x); uo_[2] = make_float2(Ul.y, Ul.z);
        invo = inv; uo = u;
    };
    // (IA, pA) of a link are shifted to the parent's pivot IN PLACE once the link's own dofs are eliminated (the link no longer needs them about
    // its own pivot), so that the parent reads them straight out of the child's registers: no second copy of the 21 + 6 values is alive.
#pragma unroll 1
    for (int lv = dmax; lv >= 0; --lv) {
        if (dlev == lv) {
            if (c.ndof == 3) { eliminate(S2, g2, 2, inv2, u2); eliminate(S1, g1, 1, inv1, u1); }
            if (c.ndof >= 1) eliminate(S0, g0, 0, inv0, u0);
            // express (IA, pA) about the parent's reference point: shift by c = cw:  B' = B + C V ; A' = A - B C + C B'^T   (C = [c]x)
            const V3 v0 = mk3(IA.vv[0], IA.vv[1], IA.vv[2]), v1 = mk3(IA.vv[1], IA.vv[3], IA.vv[4]), v2 = mk3(IA.vv[2], IA.vv[4], IA.vv[5]);   // columns (= rows) of V
            const V3 b0 = mk3(IA.wv[0], IA.wv[1], IA.wv[2]), b1 = mk3(IA.wv[3], IA.wv[4], IA.wv[5]), b2 = mk3(IA.wv[6], IA.wv[7], IA.wv[8]);   // rows of B
            const V3 k0 = cross(cw, v0), k1 = cross(cw, v1), k2 = cross(cw, v2);   // columns of C V
            const V3 n0 = mk3(b0.x + k0.x, b0.y + k1.x, b0.z + k2.x), n1 = mk3(b1.x + k0.y, b1.y + k1.y, b1.z + k2.y), n2 = mk3(b2.x + k0.z, b2.y + k1.z, b2.z + k2.z);   // rows of B'
            const V3 p0 = cross(b0, cw), p1 = cross(b1, cw), p2 = cross(b2, cw);   // rows of B C
            const V3 q0 = cross(cw, n0), q1 = cross(cw, n1), q2 = cross(cw, n2);   // columns of C B'^T
            IA.ww[0] += q0.x - p0.x; IA.ww[1] += q1.x - p0.y; IA.ww[2] += q2.x - p0.z;
            IA.ww[3] += q1.y - p1.y; IA.ww[4] += q2.y - p1.z; IA.ww[5] += q2.z - p2.z;
            IA.wv[0] = n0.x; IA.wv[1] = n0.y; IA.wv[2] = n0.z; IA.wv[3] = n1.x; IA.wv[4] = n1.y; IA.wv[5] = n1.z; IA.wv[6] = n2.x; IA.wv[7] = n2.y; IA.wv[8] = n2.z;
            pA = shift_f(pA, cw);
            // children -> parent through the environment's scratch (the Y block of the constraint rows, not live during this routine): the link
            // publishes its shifted (IA, pA) as 7 float4, its parent adds its children's in child order.  (Was 33 shuffles + 33 predicated
            // adds per child slot of the level.)
            float4* o4 = reinterpret_cast<float4*>(scr + c.lane * 28);
            o4[0] = make_float4(IA.ww[0], IA.ww[1], IA.ww[2], IA.ww[3]); o4[1] = make_float4(IA.ww[4], IA.ww[5], IA.wv[0], IA.wv[1]);
            o4[2] = make_float4(IA.wv[2], IA.wv[3], IA.wv[4], IA.wv[5]); o4[3] = make_float4(IA.wv[6], IA.wv[7], IA.wv[8], IA.vv[0]);
            o4[4] = make_float4(IA.vv[1], IA.vv[2], IA.vv[3], IA.vv[4]); o4[5] = make_float4(IA.vv[5], pA.a.x, pA.a.y, pA.a.z);
            o4[6] = make_float4(pA.l.x, pA.l.y, pA.l.z, 0.f);
        }
        __syncwarp();
        if (dlev == lv - 1) {   // lv == 0: the root's lane gathers the base's children
#pragma unroll 1
            for (int k = 0; k < dnch; ++k) {
                const float4* i4 = reinterpret_cast<const float4*>(scr + ((dchild >> (8 * k)) & 0xff) * 28);
                const float4 g0 = i4[0], g1 = i4[1], g2 = i4[2], g3 = i4[3], g4 = i4[4], g5 = i4[5], g6 = i4[6];
                IA.ww[0] += g0.x; IA.ww[1] += g0.y; IA.ww[2] += g0.z; IA.ww[3] += g0.w; IA.ww[4] += g1.x; IA.ww[5] += g1.y;
                IA.wv[0] += g1.z; IA.wv[1] += g1.w; IA.wv[2] += g2.x; IA.wv[3] += g2.y; IA.wv[4] += g2.z; IA.wv[5] += g2.w; IA.wv[6] += g3.x; IA.wv[7] += g3.y; IA.wv[8] += g3.z;
                IA.vv[0] += g3.w; IA.vv[1] += g4.x; IA.vv[2] += g4.y; IA.vv[3] += g4.z; IA.vv[4] += g4.w; IA.vv[5] += g5.x;
                pA.a.x += g5.y; pA.a.y += g5.z; pA.a.z += g5.w; pA.l.x += g6.x; pA.l.y += g6.y; pA.l.z += g6.z;
            }
        }
    }
    // ---- base: the (massless) floating base carries the root link's inertia and everything gathered on the root's lane, about the base origin in
    // world axes: Cholesky of the 6x6 directly in the generalised base coordinates [omega_w, v_w]
    S6 aB = mks(mk3(0, 0, 0), mk3(0, 0, 0));
    if (c.lane == 0) {
        float a[6][6];   // lower triangle a[i][j], j <= i ; coordinates [w(3); v(3)]
        a[0][0] = IA.ww[0]; a[1][0] = IA.ww[1]; a[1][1] = IA.ww[3]; a[2][0] = IA.ww[2]; a[2][1] = IA.ww[4]; a[2][2] = IA.ww[5];
        a[3][0] = IA.wv[0]; a[3][1] = IA.wv[3]; a[3][2] = IA.wv[6]; a[4][0] = IA.wv[1]; a[4][1] = IA.wv[4]; a[4][2] = IA.wv[7]; a[5][0] = IA.wv[2]; a[5][1] = IA.wv[5]; a[5][2] = IA.wv[8];   // B'^T
        a[3][3] = IA.vv[0]; a[4][3] = IA.vv[1]; a[4][4] = IA.vv[3]; a[5][3] = IA.vv[2]; a[5][4] = IA.vv[4]; a[5][5] = IA.vv[5];
        float gi[6];   // 1 / G_ii
#pragma unroll
        for (int j = 0; j < 6; ++j) {
            float d = a[j][j];
#pragma unroll
            for (int k = 0; k < j; ++k) d -= a[j][k] * a[j][k];
            gi[j] = rsqrtf(d);
            a[j][j] = d * gi[j];
#pragma unroll
            for (int i = j + 1; i < 6; ++i) {
                float s = a[i][j];
#pragma unroll
                for (int k = 0; k < j; ++k) s -= a[i][k] * a[j][k];
                a[i][j] = s * gi[j];
            }
        }
        // x = -(G G^T)^-1 p
        float x[6] = {-pA.a.x, -pA.a.y, -pA.a.z, -pA.l.x, -pA.l.y, -pA.l.z};
#pragma unroll
        for (int i = 0; i < 6; ++i) {
#pragma unroll
            for (int k = 0; k < i; ++k) x[i] -= a[i][k] * x[k];
            x[i] *= gi[i];
        }
#pragma unroll
        for (int i = 5; i >= 0; --i) {
#pragma unroll
            for (int k = i + 1; k < 6; ++k) x[i] -= a[k][i] * x[k];
            x[i] *= gi[i];
        }
        aB = mks(mk3(x[0], x[1], x[2]), mk3(x[3], x[4], x[5]));
        if (bullet) {   // factor kept for the constraint rows: strict lower part (15) + reciprocal diagonal (6); base velocity += h * acceleration
            int o = 0;
#pragma unroll
            for (int i = 1; i < 6; ++i)
#pragma unroll
                for (int k = 0; k < i; ++k) sG[o++] = a[i][k];
#pragma unroll
            for (int i = 0; i < 6; ++i) sG[15 + i] = gi[i];
#pragma unroll
            for (int i = 0; i < 6; ++i) sB[7 + i] = cl100(sB[7 + i] + h * x[i]);
        }
        if (DEBUG && dbg_acc) for (int i = 0; i < 6; ++i) dbg_acc[i] = x[i];
    }
    // ---- accelerations (root -> leaves): qdd_d = (u_d - U_d . a') / D_d
    float qd0 = 0.f, qd1 = 0.f, qd2 = 0.f;
    S6 al = mks(mk3(0, 0, 0), mk3(0, 0, 0));   // link acceleration (deviation from the bias acceleration)
    // U of this link's dofs back into registers (the articulated inertia is dead by now): the recursion below then has no shared-memory load on its chain
    float ur[18];
    {
        const float4* u4 = reinterpret_cast<const float4*>(uown);
        const float4 a0 = u4[0], a1 = u4[1], a2 = u4[2], a3 = u4[3];
        const float2 a4 = *reinterpret_cast<const float2*>(uown + 16);
        ur[0] = a0.x; ur[1] = a0.y; ur[2] = a0.z; ur[3] = a0.w; ur[4] = a1.x; ur[5] = a1.y; ur[6] = a1.z; ur[7] = a1.w; ur[8] = a2.x; ur[9] = a2.y; ur[10] = a2.z; ur[11] = a2.w;
        ur[12] = a3.x; ur[13] = a3.y; ur[14] = a3.z; ur[15] = a3.w; ur[16] = a4.x; ur[17] = a4.y;
    }
    auto udot = [&](S6 a, int d) { const float* q_ = ur + 6 * d; return a.a.x * q_[0] + a.a.y * q_[1] + a.a.z * q_[2] + a.l.x * q_[3] + a.l.y * q_[4] + a.l.z * q_[5]; };
    auto descend = [&](S6 a) {
        if (c.ndof >= 1) { qd0 = inv0 * (u0 - udot(a, 0)); a.a += qd0 * S0; }
        if (c.ndof == 3) { qd1 = inv1 * (u1 - udot(a, 1)); a.a += qd1 * S1; qd2 = inv2 * (u2 - udot(a, 2)); a.a += qd2 * S2; }
        return a;
    };
    if (isroot) al = aB;   // at the base origin; the root link has no dofs
#pragma unroll 1
    for (int lv = 0; lv <= dmax; ++lv) {
        S6 pa = T::shfl6(al, dpar);
        if (dlev == lv) al = descend(shift_m(pa, cw));
    }
    if (bullet) {
        // links without a level of their own move with their kinematic parent: the root link (its pivot is offset from the base origin) and the
        // lumped leaves get the parent's acceleration at their own pivot
        const S6 pk = T::shfl6(al, c.plane);
        if (isroot || dlev == 100) al = shift_m(pk, cwk);
        if (c.act) {   // publish the factors and the advanced link velocity (linear in the generalised velocities; the clamp only acts on exploding states)
            float* u = sU + c.lane * 24;   // U0 U1 U2 are already there (eliminate)
            *reinterpret_cast<float2*>(u + 18) = make_float2(inv0, inv1);
            *reinterpret_cast<float4*>(u + 20) = make_float4(inv2, sqrtf(inv0), sqrtf(inv1), sqrtf(inv2));
            float* v = sV + c.lane * 12;
            *reinterpret_cast<float4*>(v) = make_float4(velk.a.x + h * al.a.x, velk.a.y + h * al.a.y, velk.a.z + h * al.a.z, velk.l.x + h * al.l.x);
            *reinterpret_cast<float2*>(v + 4) = make_float2(velk.l.y + h * al.l.y, velk.l.z + h * al.l.z);
        }
    }
    __syncwarp();
    return make_float3(qd0, qd1, qd2);
}

// Velocity correction of the constraint impulses: dv = L^-1 D^-1/2 z with z = Y^T lambda (sZ), by the root -> leaves pass over the factors
// published by aba_solve.  Lane 0 also corrects the base velocity in sB.  Returns this link's joint-rate corrections.
template <int W>
__device__ __noinline__ float3 dv_pass() {
    const Ctx c = make_ctx<W>();
    using T = Tl<W>;
    const StepLayout& LY = lay_of(c);
    const float* sU = c.E + LY.oU; const float* sS = c.E + LY.oR; float* sG = c.E + LY.oG; float* sB = sG + 21; const float* sZ = c.E + LY.oZ;
    float q[12], u[24];
    ld12(sS + c.li * 12, q); ld12(sU + c.li * 24, u); ld12(sU + c.li * 24 + 12, u + 12);
    const V3 S0 = mk3(q[0], q[1], q[2]), S1 = mk3(q[3], q[4], q[5]), S2 = mk3(q[6], q[7], q[8]);
    V3 cw = mk3(q[9], q[10], q[11]);
    const int dof0 = reinterpret_cast<const int*>(c.LK + c.li * kLkFloats)[kLInt2] & 0xff;
    // dynamics tree (as in aba_solve): the root's lane carries the base's correction at the base origin, its children shift by both pivot offsets
    const int dyn = c.act ? reinterpret_cast<const int*>(c.LK + c.li * kLkFloats)[kLDyn] : (100 << 8);
    const int dpar = dyn & 0xff, dlev = static_cast<int>(static_cast<signed char>((dyn >> 8) & 0xff)), byp = (dyn >> 16) & 0xff;
    const int dmax = reinterpret_cast<const int*>(step_smem())[kHDmax];
    if (byp != 0xff) { const float* qb = sS + byp * 12; cw = cw + mk3(qb[9], qb[10], qb[11]); }
    S6 dB = mks(mk3(0, 0, 0), mk3(0, 0, 0));
    if (c.lane == 0) {   // base: dB = G^-T z
        float x[6] = {sZ[0], sZ[1], sZ[2], sZ[3], sZ[4], sZ[5]};
        float g[15];
#pragma unroll
        for (int k = 0; k < 15; ++k) g[k] = sG[k];
#pragma unroll
        for (int i = 5; i >= 0; --i) {
#pragma unroll
            for (int k = i + 1; k < 6; ++k) x[i] -= g[k * (k - 1) / 2 + i] * x[k];
            x[i] *= sG[15 + i];
        }
        dB = mks(mk3(x[0], x[1], x[2]), mk3(x[3], x[4], x[5]));
#pragma unroll
        for (int i = 0; i < 6; ++i) sB[7 + i] = cl100(sB[7 + i] + x[i]);
    }
    float z0 = 0.f, z1 = 0.f, z2 = 0.f, qd0 = 0.f, qd1 = 0.f, qd2 = 0.f;
    if (c.ndof >= 1) z0 = sZ[dof0] * u[21];
    if (c.ndof == 3) { z1 = sZ[dof0 + 1] * u[22]; z2 = sZ[dof0 + 2] * u[23]; }
    auto descend = [&](S6 a) {
        if (c.ndof >= 1) { qd0 = z0 - u[18] * (a.a.x * u[0] + a.a.y * u[1] + a.a.z * u[2] + a.l.x * u[3] + a.l.y * u[4] + a.l.z * u[5]); a.a += qd0 * S0; }
        if (c.ndof == 3) {
            qd1 = z1 - u[19] * (a.a.x * u[6] + a.a.y * u[7] + a.a.z * u[8] + a.l.x * u[9] + a.l.y * u[10] + a.l.z * u[11]); a.a += qd1 * S1;
            qd2 = z2 - u[20] * (a.a.x * u[12] + a.a.y * u[13] + a.a.z * u[14] + a.l.x * u[15] + a.l.y * u[16] + a.l.z * u[17]); a.a += qd2 * S2;
        }
        return a;
    };
    S6 al = mks(mk3(0, 0, 0), mk3(0, 0, 0));
    if (c.lane == 0) al = dB;
#pragma unroll 1
    for (int lv = 0; lv <= dmax; ++lv) {
        S6 pa = T::shfl6(al, dpar);
        if (dlev == lv) al = descend(shift_m(pa, cw));
    }
    __syncwarp();
    return make_float3(qd0, qd1, qd2);
}

// Link velocities from the generalised velocities (root -> leaves), for the environments flagged by `want`.  Only needed when Bullet's
// per-coordinate velocity clamp (maxCoordinateVelocity = 100) fired in the velocity update: otherwise aba_solve's v + h a is the same thing.
template <int W>
__device__ __noinline__ void vel_pass(float jvx, float jvy, float jvz, bool want) {
    const Ctx c = make_ctx<W>();
    using T = Tl<W>;
    const StepLayout& LY = lay_of(c);
    const float* sS = c.E + LY.oR; float* sV = c.E + LY.oV; const float* sB = c.E + LY.oG + 21;
    float q[12];
    ld12(sS + c.li * 12, q);
    const V3 S0 = mk3(q[0], q[1], q[2]), S1 = mk3(q[3], q[4], q[5]), S2 = mk3(q[6], q[7], q[8]), cw = mk3(q[9], q[10], q[11]);
    V3 jww = mk3(0, 0, 0);
    if (c.jtype == kJSpherical) jww = jvx * S0 + jvy * S1 + jvz * S2; else if (c.jtype == kJRevolute) jww = jvx * S0;
    S6 vel = mks(mk3(0, 0, 0), mk3(0, 0, 0));
    if (c.lane == 0) { const V3 bo = mk3(sB[7], sB[8], sB[9]); vel = mks(bo + jww, mk3(sB[10], sB[11], sB[12]) + cross(bo, cw)); }
#pragma unroll 1
    for (int lv = 1; lv <= c.maxlevel; ++lv) {
        const S6 pv = T::shfl6(vel, c.plane);
        if (c.level == lv) vel = mks(pv.a + jww, pv.l + cross(pv.a, cw));
    }
    if (c.act && want) {
        float* v = sV + c.lane * 12;
        v[0] = vel.a.x; v[1] = vel.a.y; v[2] = vel.a.z; v[3] = vel.l.x; v[4] = vel.l.y; v[5] = vel.l.z;
    }
    __syncwarp();
}

// VAR selects optional scene features compiled into separate instantiations so that the plain imitate kernel carries none of their code:
//   bit 0 (kVarTask)    AMP task scenes: task block advanced after every update (dm_task.cuh)
//   bit 1 (kVarRootRot) --sync_char_root_rot: the heading sync of cSceneImitate::SyncKinCharNewCycle at a clip wrap
template <int W, bool DEBUG, int VAR>
__global__ void __launch_bounds__(kStepMaxThreads, 1) dm_step_kernel(const DevModel* __restrict__ gm, DevState st, const double* __restrict__ frame_times,
                                                                       const float* __restrict__ frames, double dt, int n_updates, int sim_substeps, StepLayout LY) {
    constexpr bool TASK = (VAR & kVarTask) != 0, ROOTROT = (VAR & kVarRootRot) != 0;
    using T = Tl<W>;
    extern __shared__ __align__(16) float sm[];
    const int tiles = blockDim.x / W;
    const int tile = threadIdx.x / W;
    const int lane = threadIdx.x % W;
    const int env = blockIdx.x * tiles + tile;   // host guarantees num_envs (padded) is a multiple of tiles
    const DevModel& M = *gm;
    const int nl = LY.nl, CL = LY.chain_len;
    const bool act = lane < nl;
    const int li = act ? lane : nl - 1;

    // ---- block-shared header (layout, children per level, launch constants) and tables: per-link constants (LK), common chain depth of two
    // links (CD), chain depth -> dof (CH)
    float* LK = sm + kHdrFloats;
    unsigned char* CD = reinterpret_cast<unsigned char*>(LK + nl * kLkFloats);
    unsigned char* CH = CD + nl * nl;
    int* LYS = reinterpret_cast<int*>(sm + kHLayout);   // shared copy of the layout for the phase routines
    for (int j = threadIdx.x; j < nl; j += blockDim.x) {
        const DevLink& K = M.link[j];
        float* q = LK + j * kLkFloats;
        const int p = K.parent;
        for (int k = 0; k < 3; ++k) { q[kLC + k] = K.evec[k] + (p >= 0 ? M.link[p].dvec[k] : 0.f); q[kLD + k] = K.dvec[k]; q[kLAx + k] = K.axis[k]; }
        q[kLM] = K.mass;
        // ---- dynamics tree of the articulated-body passes (aba_solve, dv_pass).  Links without dofs need no level of their own there:
        //   * the root link is fixed to the floating base: its rigid inertia is referred to the BASE ORIGIN (constant in link axes), its lane
        //     accumulates the base's 6 x 6, and its children hang off the base directly (their shift is the sum of the two pivot offsets),
        //   * a fixed leaf (humanoid3d: the wrists) is lumped into its parent: mass, first moment and inertia of the pair about the parent's
        //     pivot are constants in the parent's axes.
        // Same rigid-body system, two tree levels fewer (humanoid3d: 5 -> 3) in every pass of those routines.  The kinematic tree (kin_pass,
        // the constraint rows' chain walks, vel_pass) is unchanged.
        auto lumped = [&](int c_) { const DevLink& C_ = M.link[c_]; return C_.ndof == 0 && C_.nchild == 0 && C_.parent >= 0 && M.link[C_.parent].ndof > 0; };
        const bool isroot = p < 0, self_lumped = lumped(j);
        {
            // composite rigid body about the reference point (COM of part i at r_i): ww = sum Icom_i + m_i (|r_i|^2 1 - r_i r_i^T), first moment sum m_i r_i
            float cm = 0.f, mdx = 0.f, mdy = 0.f, mdz = 0.f, wD[6] = {0, 0, 0, 0, 0, 0}, wB[6] = {0, 0, 0, 0, 0, 0};
            auto add_part = [&](float m_, V3 r, const float* iD, const float* iB) {   // iD / iB: symmetric 3 x 3 about the part's COM, this link's axes
                const float rr = dot(r, r);
                const float sh[6] = {m_ * (rr - r.x * r.x), -m_ * r.x * r.y, -m_ * r.x * r.z, m_ * (rr - r.y * r.y), -m_ * r.y * r.z, m_ * (rr - r.z * r.z)};
                for (int k = 0; k < 6; ++k) { wD[k] += iD[k] + sh[k]; wB[k] += iB[k] + sh[k]; }
                cm += m_; mdx += m_ * r.x; mdy += m_ * r.y; mdz += m_ * r.z;
            };
            if (!self_lumped) {
                V3 r = mk3(K.dvec[0], K.dvec[1], K.dvec[2]);
                if (isroot) r = r + mul(qmat(mkq(K.zrot[0], K.zrot[1], K.zrot[2], K.zrot[3])), mk3(K.evec[0], K.evec[1], K.evec[2]));   // base origin -> pivot, link axes
                const float iD[6] = {K.inertiaD[0], 0.f, 0.f, K.inertiaD[1], 0.f, K.inertiaD[2]}, iB[6] = {K.inertiaB[0], 0.f, 0.f, K.inertiaB[1], 0.f, K.inertiaB[2]};
                add_part(K.mass, r, iD, iB);
                for (int k = 0; k < K.nchild; ++k) {
                    const int c_ = K.child[k];
                    if (!lumped(c_)) continue;
                    const DevLink& C_ = M.link[c_];
                    const M3 Rc = qmat(mkq(C_.zrot[0], C_.zrot[1], C_.zrot[2], C_.zrot[3]));   // this link's axes -> the child's axes (fixed joint)
                    const V3 rc = mk3(C_.evec[0] + K.dvec[0], C_.evec[1] + K.dvec[1], C_.evec[2] + K.dvec[2]) + mulT(Rc, mk3(C_.dvec[0], C_.dvec[1], C_.dvec[2]));
                    const float cD[6] = {C_.inertiaD[0], 0.f, 0.f, C_.inertiaD[1], 0.f, C_.inertiaD[2]}, cB[6] = {C_.inertiaB[0], 0.f, 0.f, C_.inertiaB[1], 0.f, C_.inertiaB[2]};
                    float rD[6], rB[6];
                    rot_sym(Rc, cD, rD); rot_sym(Rc, cB, rB);
                    add_part(C_.mass, rc, rD, rB);
                }
            }
            for (int k = 0; k < 6; ++k) { q[kLWd + k] = wD[k]; q[kLWb + k] = wB[k]; }
            q[kLMc] = cm;
            const float icm = cm > 0.f ? 1.0f / cm : 0.f;
            q[kLDc] = mdx * icm; q[kLDc + 1] = mdy * icm; q[kLDc + 2] = mdz * icm;
            int dch = 0, dn = 0;
            for (int k = 0; k < K.nchild; ++k) if (!lumped(K.child[k])) { dch |= (K.child[k] & 0xff) << (8 * dn); ++dn; }
            const int dlev = isroot ? -1 : (self_lumped ? 100 : K.level - 1);
            const int dpar = isroot ? 0 : p, byp = (!isroot && p >= 0 && M.link[p].parent < 0) ? p : 0xff;
            reinterpret_cast<int*>(q)[kLDyn] = (dpar & 0xff) | ((dlev & 0xff) << 8) | ((byp & 0xff) << 16) | ((dn & 0xff) << 24);
            reinterpret_cast<int*>(q)[kLDChild] = dch;
        }
        reinterpret_cast<int*>(q)[kLInt] = (K.parent & 0xff) | ((K.jtype & 0xff) << 8) | ((K.ndof & 0xff) << 16) | ((K.depth0 & 0xff) << 24);
        reinterpret_cast<int*>(q)[kLInt2] = (K.dof0 & 0xff) | ((K.last_depth & 0xff) << 8) | ((K.nchild & 0xff) << 16);
        for (int k = 0; k < 4; ++k) q[kLZr + k] = K.zrot[k];
        for (int k = 0; k < 3; ++k) q[kLHe + k] = K.he[k];
        q[kLThr] = K.break_thr; q[kLKp] = K.kp; q[kLKd] = K.kd; q[kLTl] = K.tlim; q[kLLo] = K.lim_lo; q[kLHi] = K.lim_hi;
        reinterpret_cast<int*>(q)[kLFlg] = (K.shape & 0xff) | ((K.fall_contact & 0xff) << 8) | ((K.has_limit & 0xff) << 16);
        reinterpret_cast<int*>(q)[kLTree] = (K.level & 0xff) | ((M.maxlevel & 0xff) << 8) | ((K.nchild & 0xff) << 16);
        reinterpret_cast<int*>(q)[kLChild] = (K.child[0] & 0xff) | ((K.child[1] & 0xff) << 8) | ((K.child[2] & 0xff) << 16) | ((K.child[3] & 0xff) << 24);
        for (int d = 0; d < CL; ++d) CH[j * CL + d] = M.chain_dof[j][d];
        for (int b = 0; b < nl; ++b) {
            int cnt = 0;
            const int lim = min(K.last_depth, M.link[b].last_depth);
            while (cnt <= lim && M.chain_dof[j][cnt] == M.chain_dof[b][cnt]) ++cnt;
            CD[j * nl + b] = static_cast<unsigned char>(cnt);
        }
    }
    if (threadIdx.x == blockDim.x - 1) {
        static_assert(sizeof(StepLayout) / sizeof(int) <= kHLvc, "StepLayout must fit the header slot");
        const int* src = reinterpret_cast<const int*>(&LY);
        for (int k = 0; k < static_cast<int>(sizeof(StepLayout) / sizeof(int)); ++k) LYS[k] = src[k];
        sm[kHGrav] = M.gravity[0]; sm[kHGrav + 1] = M.gravity[1]; sm[kHGrav + 2] = M.gravity[2];
        sm[kHh] = static_cast<float>(dt) / static_cast<float>(sim_substeps); sm[kHScale] = M.scale; sm[kHMu] = M.friction; sm[kHFdt] = static_cast<float>(dt);
    }
    if (threadIdx.x == 8) {   // deepest level of the dynamics tree (levels of the links with dofs, the root's children being level 0)
        int mx = 0;
        for (int j = 0; j < nl; ++j) { const DevLink& K = M.link[j]; if (K.parent >= 0 && !(K.ndof == 0 && K.nchild == 0 && M.link[K.parent].ndof > 0)) mx = max(mx, K.level - 1); }
        reinterpret_cast<int*>(sm)[kHDmax] = mx;
    }
    __syncthreads();

    float* E = sm + LY.hot_floats + tile * LY.env_floats;
    // every word of the environment's block is initialised once per launch: the constraint sweeps read (and discard) words past the live rows
    // of a section, which must hold finite numbers (a NaN pattern left by an earlier kernel would survive the multiplication by a zero update)
    for (int k = lane * 4; k < LY.env_floats; k += W * 4) *reinterpret_cast<float4*>(E + k) = make_float4(0.f, 0.f, 0.f, 0.f);
    __syncwarp();
    float* sV = E + LY.oV; float* sG = E + LY.oG; float* sQ = E + LY.oQ; float* sLam = E + LY.oLam;
    const float* LKo = LK + li * kLkFloats;
    const int jtype = (reinterpret_cast<const int*>(LKo)[kLInt] >> 8) & 0xff, ndof = act ? ((reinterpret_cast<const int*>(LKo)[kLInt] >> 16) & 0xff) : 0;
    const int dof0 = reinterpret_cast<const int*>(LKo)[kLInt2] & 0xff;
    const int lflags = reinterpret_cast<const int*>(LKo)[kLFlg];
    const bool fall_contact = ((lflags >> 8) & 0xff) != 0, has_limit = ((lflags >> 16) & 0xff) != 0;

    // ---- state load (env-major block, float4)
    const int ss = sim_stride(nl);
    float* sim = st.sim + static_cast<size_t>(env) * ss;
    double* tm = st.time + static_cast<size_t>(env) * kTimeDoubles;
    int* fl = st.flags + static_cast<size_t>(env) * kFlagInts;
    float* mani = st.manifold + static_cast<size_t>(env) * nl * kManifoldFloats;
    // AMP task scenes (TASK instantiations only): the environment's task block, advanced by lane 0 after every update (dm_task.cuh)
    double* tk = nullptr;
    double* tkx = nullptr;
    if constexpr (TASK) { tk = st.task + static_cast<size_t>(env) * kTaskDoubles; tkx = st.taskx + static_cast<size_t>(env) * kTaskExtDoubles; }
    float* sB = sG + 21;   // base state, owned by lane 0: position [0..2], quaternion (world->base) [3..6], omega_w [7..9], v_w [10..12]
    if (lane == 0) {
        float4 b0 = reinterpret_cast<const float4*>(sim)[0], b1 = reinterpret_cast<const float4*>(sim)[1], b2 = reinterpret_cast<const float4*>(sim)[2],
               b3 = reinterpret_cast<const float4*>(sim)[3];
        sB[0] = b0.x; sB[1] = b0.y; sB[2] = b0.z; sB[3] = b1.x; sB[4] = b1.y; sB[5] = b1.z; sB[6] = b1.w;
        sB[7] = b2.x; sB[8] = b2.y; sB[9] = b2.z; sB[10] = b3.x; sB[11] = b3.y; sB[12] = b3.z;
    }
    float4 jp = reinterpret_cast<const float4*>(sim + 16)[li];
    float4 jv = reinterpret_cast<const float4*>(sim + 16 + 4 * nl)[li];
    // the f64 clocks (timer, mocap time, controller time, origin) live in global memory and are advanced in place by lane 0 once per update;
    // cbits carries what the post-update flags need: bit 0 new-action edge, bit 1 time limit reached, bit 2 non-looping clip finished
    int need_action = fl[kFNeedAction];
    int cbits = 0;
    bool alive = fl[kFDone] == 0;
    int f_over = fl[kFRowOverflow], f_updates = fl[kFUpdates];
    __syncwarp();

    const float h = static_cast<float>(dt) / static_cast<float>(sim_substeps);
    const float fdt = static_cast<float>(dt);
    const float gx = M.gravity[0], gy = M.gravity[1], gz = M.gravity[2];
    const float scale = M.scale, mu = M.friction;
    float* dbg = (DEBUG && st.pdbg) ? st.pdbg + static_cast<size_t>(env) * kDebugFloats : nullptr;   // test hook: stage dumps of the first update

    float tau0 = 0.f, tau1 = 0.f, tau2 = 0.f;   // joint torques of the current update (body-frame components / revolute scalar)
    bool in_contact_tol = false;

#ifdef DM_PROFILE
    // per-warp cycle counters per code section (profile build only): lane 0 accumulates, written to st.pdbg at the end
    unsigned int* PRF = reinterpret_cast<unsigned int*>(sm + LY.hot_floats + tiles * LY.env_floats) + (threadIdx.x / 32) * 16;
    if ((threadIdx.x & 31) == 0) for (int k = 0; k < 16; ++k) PRF[k] = 0u;
    unsigned int prf_t = static_cast<unsigned int>(clock64());
#define PROF(sec) do { if ((threadIdx.x & 31) == 0) { unsigned int t_ = static_cast<unsigned int>(clock64()); PRF[sec] += t_ - prf_t; prf_t = t_; } } while (0)
    unsigned int* PRFP = PRF;
#else
#define PROF(sec) do { } while (0)
    unsigned int* PRFP = nullptr;
#endif
    bool need_kin = true, pending_flags = false;
    int mcnt = 4;   // cached points of this lane's link after the last collision pass; unknown at the start of a launch: forces the first read
    const int stages_per_upd = sim_substeps + 1;
    const int total_stages = n_updates * stages_per_upd;
#pragma unroll 1
    for (int stage = 0; stage <= total_stages; ++stage) {
        // the manifold of this lane's link is read by the collision pass of a Bullet sub-step: start pulling its two cache lines in now
        if ((stage % stages_per_upd) != 0 && act && alive && mcnt > 0) {
            const float* mp_ = mani + li * kManifoldFloats;
            asm volatile("prefetch.global.L1 [%0];" ::"l"(mp_));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(mp_ + 32));
        }
        // =================================================================== forward kinematics + link velocities
        if (need_kin) { need_kin = false; kin_pass<W>(jp, jv); }
        PROF(0);
        // =================================================================== post-update flags of the update that just finished
        if (pending_flags) {
            pending_flags = false;
            need_action = cbits & 1;
            // fall: any fall-contact link with a manifold point at distance <= 0.001*scale (state of the last sub-step's collision pass)
            const unsigned fb = __ballot_sync(0xffffffffu, act && fall_contact && in_contact_tol);
            const unsigned fseg = (W == 32) ? fb : ((fb >> (threadIdx.x & 16)) & 0xffffu);
            const int fallen = (fseg != 0 && M.enable_contact_fall) ? 1 : 0;
            // exploded velocities: any link |v|, |w| component > 100 in world axes (cSimCharacter::HasVelExploded); v at the COM
            const float* v = sV + li * 12;
            const V3 wa = mk3(v[0], v[1], v[2]);
            const V3 vw = (mk3(v[3], v[4], v[5]) + cross(wa, mk3(v[6], v[7], v[8]))) * (1.0f / scale);
            float mx = fmaxf(fmaxf(fmaxf(fabsf(vw.x), fabsf(vw.y)), fabsf(vw.z)), fmaxf(fmaxf(fabsf(wa.x), fabsf(wa.y)), fabsf(wa.z)));
            const unsigned eb = __ballot_sync(0xffffffffu, act && mx > 100.f);
            const unsigned eseg = (W == 32) ? eb : ((eb >> (threadIdx.x & 16)) & 0xffffu);
            int task_fail = 0;          // 0 none, 1 fail, 2 success (cRLScene::eTerminate)
            int fallen_eff = fallen;    // HasFallen as the scene sees it (the get-up scene ignores contacts while getting up)
            if constexpr (TASK) {
                // cSceneTargetAMP::Update: target timer / position / heading / speed after the scene update, then the distance failure of
                // CheckTerminate; the COM is kept for CalcReward (SceneTargetAMP.cpp:3-80,136-145,294-319).  heading_amp_getup and strike_amp
                // (dm_task_ext.cuh) additionally need a few bodies' positions / velocities, published to lane 0 by shuffles.
                const V3 com = tile_com<W>(E + LY.oW + li * 12, v, act ? LKo[kLM] : 0.f, 1.0f / (M.total_mass * scale));
                const int kind = M.task_kind;
                TaskBodies B;
                if (kind >= kTaskHeadingGetup) {
                    const float* w_ = E + LY.oW + li * 12;
                    const V3 cpos = mk3((w_[9] + v[6]) / scale, (w_[10] + v[7]) / scale, (w_[11] + v[8]) / scale);   // this lane's body COM, unscaled
                    const TaskExtParams& X = M.taskx;
                    B.head_y = T::shfl(cpos.y, X.head_id);
                    B.contact_fall = fallen;
#pragma unroll
                    for (int k = 0; k < kMaxTaskBodies; ++k) {
                        const V3 sp = T::shfl3(cpos, k < X.n_strike ? X.strike_bodies[k] : 0), sv = T::shfl3(vw, k < X.n_strike ? X.strike_bodies[k] : 0);
                        const V3 fp = T::shfl3(cpos, k < X.n_fail ? X.fail_bodies[k] : 0);
                        B.spos[k][0] = sp.x; B.spos[k][1] = sp.y; B.spos[k][2] = sp.z; B.svel[k][0] = sv.x; B.svel[k][1] = sv.y; B.svel[k][2] = sv.z;
                        B.fpos[k][0] = fp.x; B.fpos[k][1] = fp.y; B.fpos[k][2] = fp.z;
                    }
                }
                int tf = 0, fe = fallen;
                if (lane == 0 && alive) {
                    TaskRng rng{M.task_seed, M.env_id_base + static_cast<unsigned long long>(env), tk + kKCounter};
                    const double rx = static_cast<double>(sB[0]) / M.scale, rz = static_cast<double>(sB[2]) / M.scale;
                    tk[kKCom] = com.x; tk[kKCom + 1] = com.y; tk[kKCom + 2] = com.z;
                    if (kind == kTaskStrike) {
                        // cSceneTargetAMP::UpdateTarget without the timed re-draw (CheckTargetReset is false in this scene), hit detection,
                        // then the target timer's own restart (SceneTargetAMP.cpp:136-145; SceneStrikeAMP.cpp:289-298,385-388)
                        const double scene_time = tm[kTTimer];
                        tk[kKTimer] += dt;
                        strike_update(M.taskx, tk, tkx, rx, rz, scene_time, B);
                        if (tk[kKTimer] >= tk[kKTimerMax]) task_timer_reset(M.task, tk, rng);
                        tf = strike_terminate(M.task, M.taskx, tk, tkx, rx, rz, scene_time);
                    } else {
                        task_update(task_base_kind(kind), M.task, tk, rng, dt, rx, rz);
                        tf = task_dist_fail(kind, M.task, tk, rx, rz) ? 1 : 0;
                        if (kind == kTaskHeadingGetup) {
                            tkx[kXHeadY] = B.head_y;
                            if (getup_update(M.taskx, tkx, dt, M.test_mode != 0, fallen != 0)) fe = 0;   // HasFallenContact override while getting up
                        }
                    }
                }
                task_fail = T::shfli(tf, 0);
                fallen_eff = T::shfli(fe, 0);
            }
            if (alive) {
                int term = (M.enable_fall_end && fallen_eff) ? 1 : 0;
                if (!term && (cbits & 4)) term = 1;
                if (TASK && !term && task_fail) term = task_fail;
                f_updates++;
                const bool end = (cbits & 2) || term;
                if (end || stage == total_stages) {   // commit
                    if (lane == 0) {
                        reinterpret_cast<float4*>(sim)[0] = make_float4(sB[0], sB[1], sB[2], 0.f);
                        reinterpret_cast<float4*>(sim)[1] = make_float4(sB[3], sB[4], sB[5], sB[6]);
                        reinterpret_cast<float4*>(sim)[2] = make_float4(sB[7], sB[8], sB[9], 0.f);
                        reinterpret_cast<float4*>(sim)[3] = make_float4(sB[10], sB[11], sB[12], 0.f);
                        fl[kFNeedAction] = need_action; fl[kFDone] = end ? 1 : 0; fl[kFTerminate] = term; fl[kFValid] = (eseg == 0) ? 1 : 0; fl[kFFallen] = fallen_eff;
                        fl[kFRowOverflow] = f_over; fl[kFUpdates] = f_updates;
                    }
                    if (act) {
                        reinterpret_cast<float4*>(sim + 16)[lane] = jp;
                        reinterpret_cast<float4*>(sim + 16 + 4 * nl)[lane] = jv;
                    }
                }
                if (end) alive = false;
            }
        }
        PROF(1);
        if (stage == total_stages) break;
        // block barrier after every stage (Stable-PD stage, each Bullet sub-step): measured on a B200, 2.12 M vs 2.11 M policy steps/s with one per update,
        // 1.94 / 1.89 / 1.78 M with one every 2 / 4 updates / none (warps that drift apart thrash the instruction cache)
        if (__syncthreads_and(!alive)) break;
        PROF(2);
        if (__ballot_sync(0xffffffffu, alive) == 0u) continue;   // both environments of this warp are frozen
        const int ph = stage % stages_per_upd;      // 0: Stable-PD stage, 1..sim_substeps: Bullet sub-steps
        const bool first_upd = stage < stages_per_upd;
        if (ph == 0) {
            // ---------------- clocks: cScene::Update, cSceneImitate::UpdateKinChar, cDeepMimicCharController::UpdateCalcTau
            int cb = 0;
            if constexpr (TASK) {
                // cDeepMimicCharController::HandleNewAction (DeepMimicCharController.cpp:262-267): COM of the state the new action starts from
                if (__ballot_sync(0xffffffffu, alive && need_action) != 0u) {
                    const V3 com = tile_com<W>(E + LY.oW + li * 12, sV + li * 12, act ? LKo[kLM] : 0.f, 1.0f / (M.total_mass * scale));
                    if (lane == 0 && alive && need_action) { tk[kKPrevCom] = com.x; tk[kKPrevCom + 1] = com.y; tk[kKPrevCom + 2] = com.z; }
                }
            }
            if (lane == 0 && alive) {
                const double timer = tm[kTTimer] + dt;
                double kin_time = tm[kTKin];
                double dur_ = M.motion_dur;
                if constexpr (TASK) dur_ = st.ctab->info[st.clip[env]].dur;   // the environment's own clip of the dataset
                const double dur = dur_;
                double p0 = kin_time / dur; p0 -= floor(p0);
                kin_time += dt;
                double p1 = kin_time / dur; p1 -= floor(p1);
                if constexpr (ROOTROT) {
                    // --sync_char_root_rot instantiation: the whole wrap handling is the shared host / device routine of dm_task.cuh
                    // (checked against the oracle on the host, tests/test_task_scenes_cpu.py)
                    if (M.loop_motion && p1 < p0 && (M.sync_root_pos || M.sync_root_rot)) {
                        const double simq[4] = {static_cast<double>(sB[3]), static_cast<double>(sB[4]), static_cast<double>(sB[5]), static_cast<double>(sB[6])};
                        kin_wrap_sync(frame_times, frames, M.pose_dim, M.num_frames, M.cycle_delta, dur, kin_time, tm + kTOrigin, tm + kTOriginRot,
                                      static_cast<double>(sB[0]) / M.scale, static_cast<double>(sB[2]) / M.scale, simq, M.sync_root_pos != 0, M.sync_root_rot != 0);
                    }
                }
                if constexpr (TASK) {
                    // task scenes: same wrap handling on the environment's own clip of the dataset
                    const ClipInfo& ci = st.ctab->info[st.clip[env]];
                    if (ci.loop && p1 < p0 && M.sync_root_pos) {
                        const double simq[4] = {static_cast<double>(sB[3]), static_cast<double>(sB[4]), static_cast<double>(sB[5]), static_cast<double>(sB[6])};
                        kin_wrap_sync(frame_times + ci.frame_off, frames + static_cast<size_t>(ci.frame_off) * M.pose_dim, M.pose_dim, ci.num_frames, ci.cycle_delta, dur, kin_time,
                                      tm + kTOrigin, tm + kTOriginRot, static_cast<double>(sB[0]) / M.scale, static_cast<double>(sB[2]) / M.scale, simq, true, false);
                    }
                }
                if (!ROOTROT && !TASK && M.loop_motion && p1 < p0 && M.sync_root_pos) {
                    // SyncKinCharNewCycle: snap the clip's root x,z (at the new time) onto the simulated root
                    double org_x = tm[kTOrigin], org_z = tm[kTOrigin + 2];
                    int cyc = static_cast<int>(floor(kin_time / dur));
                    double tt = kin_time - cyc * dur;
                    int lo = 0, hi = M.num_frames - 1;   // upper_bound - 1
                    while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (frame_times[mid] <= tt) lo = mid; else hi = mid; }
                    double bl = (tt - frame_times[lo]) / (frame_times[lo + 1] - frame_times[lo]);
                    bl = fmin(fmax(bl, 0.0), 1.0);
                    const float* f0 = frames + static_cast<size_t>(lo) * M.pose_dim; const float* f1 = f0 + M.pose_dim;
                    double rx = (1 - bl) * f0[0] + bl * f1[0] + cyc * static_cast<double>(M.cycle_delta[0]);
                    double rz = (1 - bl) * f0[2] + bl * f1[2] + cyc * static_cast<double>(M.cycle_delta[2]);
                    double qw = tm[kTOriginRot], qx = tm[kTOriginRot + 1], qy = tm[kTOriginRot + 2], qz = tm[kTOriginRot + 3];
                    double ry_ = (1 - bl) * f0[1] + bl * f1[1];
                    double ux = qy * rz - qz * ry_, uy = qz * rx - qx * rz, uz = qx * ry_ - qy * rx;
                    ux *= 2; uy *= 2; uz *= 2;
                    double kx = rx + qw * ux + (qy * uz - qz * uy);
                    double kz = rz + qw * uz + (qx * uy - qy * ux);
                    double sx = static_cast<double>(sB[0]) / M.scale, sz = static_cast<double>(sB[2]) / M.scale;
                    if (M.sync_root_pos) {
                        org_x += sx - (kx + org_x);
                        org_z += sz - (kz + org_z);
                        tm[kTOrigin + 1] = 0.0;   // kin_root.y := ground_h + (kin_root.y - origin.y)  =>  origin.y returns to 0
                    }
                    tm[kTOrigin] = org_x; tm[kTOrigin + 2] = org_z;
                }
                const double ctrl_time = tm[kTCtrl] + dt;
                if (need_action) tm[kTPrevAct] = ctrl_time;
                tm[kTTimer] = timer; tm[kTKin] = kin_time; tm[kTCtrl] = ctrl_time;
                {   // cMathUtil::CheckNextInterval(dt, ctrl_time + init_time_offset, 1/30), evaluated for the flags after this update
                    const double cur = ctrl_time + tm[kTInitOff], pad = 0.001 * dt, T_ = M.query_dt;
                    int c0 = static_cast<int>(floor((cur + pad) / T_)), c1 = static_cast<int>(floor((cur + pad - dt) / T_));
                    cb = (c0 != c1) ? 1 : 0;
                }
                if (timer >= tm[kTTimerMax]) cb |= 2;
                if (M.end_at_clip_end && kin_time >= dur) cb |= 4;
            }
            cbits = T::shfli(cb, 0);
            need_action = 0;
            PROF(3);
            // ---------------- cImpPDController::CalcControlForces (ImpPDController.cpp:136-195) in the body-frame joint coordinates of the sim state
            const float4 tg = reinterpret_cast<const float4*>(sim + 16 + 8 * nl)[li];
            float e0 = 0, e1 = 0, e2 = 0;
            if (jtype == kJSpherical) {
                Q4 q = mkq(jp.x, jp.y, jp.z, jp.w);
                // pose_inc = normalize(q + dt * 0.5 * q (x) (0, w))      (cKinTree::VelToPoseDiff, KinTree.cpp:1581-1610)
                Q4 dq = qmul(q, mkq(jv.x, jv.y, jv.z, 0.f));
                Q4 qi = qnormalize(mkq(q.x + 0.5f * fdt * dq.x, q.y + 0.5f * fdt * dq.y, q.z + 0.5f * fdt * dq.z, q.w + 0.5f * fdt * dq.w));
                V3 e = quat_rotvec3(qmul(qconj(qi), mkq(tg.x, tg.y, tg.z, tg.w)));   // cKinTree::CalcVel(dt = 1) -> CalcQuaternionVelRel
                e0 = e.x; e1 = e.y; e2 = e.z;
            } else if (jtype == kJRevolute) {
                e0 = tg.x - (normalize_angle3(jp.x) + fdt * jv.x);
            }
            const float kp = LKo[kLKp], kd = LKo[kLKd];
            const float pe0 = kp * e0, pe1 = kp * e1, pe2 = kp * e2;
            const float3 qdd = aba_solve<W, DEBUG>(pe0 - kd * jv.x, pe1 - kd * jv.y, pe2 - kd * jv.z, fdt * kd, 0, jv.x, jv.y, jv.z, nullptr);
            // ---------------- torques: tau = Kp e + Kd (edot - dt a), clamped by norm (cSimBodyJoint::ClampTotalTorque, SimBodyJoint.cpp:299-307)
            float t0 = 0, t1 = 0, t2 = 0;
            if (ndof >= 1) t0 = pe0 + kd * (-jv.x - fdt * qdd.x);
            if (ndof == 3) { t1 = pe1 + kd * (-jv.y - fdt * qdd.y); t2 = pe2 + kd * (-jv.z - fdt * qdd.z); }
            const float mag = sqrtf(t0 * t0 + t1 * t1 + t2 * t2), tlim = LKo[kLTl];
            if (mag > tlim) { float s = tlim / mag; t0 *= s; t1 *= s; t2 *= s; }
            tau0 = t0; tau1 = t1; tau2 = t2;
            if (DEBUG && dbg && first_upd) {
                if (ndof >= 1) { dbg[2 * kMaxDofs + dof0] = t0; dbg[3 * kMaxDofs + dof0] = qdd.x; }
                if (ndof == 3) { dbg[2 * kMaxDofs + dof0 + 1] = t1; dbg[2 * kMaxDofs + dof0 + 2] = t2; dbg[3 * kMaxDofs + dof0 + 1] = qdd.y; dbg[3 * kMaxDofs + dof0 + 2] = qdd.z; }
                if (lane == 0) for (int k = 0; k < 6; ++k) dbg[2 * kMaxDofs + k] = 0.f;
            }
            PROF(4);
            continue;
        }
        // =================================================================== Bullet sub-step
        const int sub = ph - 1;
        int P;
        {
            const int r = collide<W>(mani, alive ? 1 : 0, mcnt);
            P = r & 0xff; in_contact_tol = ((r >> 8) & 1) != 0; if ((r >> 9) & 1) f_over = 1; mcnt = (r >> 10) & 7;
        }
        PROF(3);
        {   // unconstrained accelerations, v += a h (the base and the link velocities are advanced inside)
            float* dacc = (DEBUG && dbg && first_upd) ? dbg + (sub == 0 ? 4 * kMaxDofs : 8 * kMaxDofs + 1024) : nullptr;
            const float3 qdd = aba_solve<W, DEBUG>(tau0, tau1, tau2, 0.f, 1, jv.x, jv.y, jv.z, dacc);
            if (DEBUG && dacc) { if (ndof >= 1) dacc[dof0] = qdd.x; if (ndof == 3) { dacc[dof0 + 1] = qdd.y; dacc[dof0 + 2] = qdd.z; } }
            bool hit = false;   // a generalised velocity reached Bullet's clamp: the link velocities must be rebuilt from the clamped values
            if (ndof >= 1) { const float v = jv.x + h * qdd.x; jv.x = cl100(v); hit |= fabsf(v) > 100.f; }
            if (ndof == 3) { const float v1 = jv.y + h * qdd.y, v2 = jv.z + h * qdd.z; jv.y = cl100(v1); jv.z = cl100(v2); hit |= fabsf(v1) > 100.f || fabsf(v2) > 100.f; }
            if (lane == 0) for (int k = 0; k < 6; ++k) hit |= fabsf(sB[7 + k]) >= 100.f;
            const unsigned hb = __ballot_sync(0xffffffffu, hit);
            if (hb != 0u) {
                const unsigned hseg = (W == 32) ? hb : ((hb >> (threadIdx.x & 16)) & 0xffffu);
                vel_pass<W>(jv.x, jv.y, jv.z, hseg != 0u);
            }
            if (DEBUG && dbg && first_upd) {
                const int o = (sub == 0 ? 5 * kMaxDofs : 9 * kMaxDofs + 1024);
                if (lane == 0) { for (int k = 0; k < 6; ++k) dbg[o + k] = sB[7 + k]; dbg[(sub == 0 ? 7 * kMaxDofs : 11 * kMaxDofs + 1024)] = static_cast<float>(P); }
                if (ndof >= 1) dbg[o + dof0] = jv.x;
                if (ndof == 3) { dbg[o + dof0 + 1] = jv.y; dbg[o + dof0 + 2] = jv.z; }
            }
        }
        PROF(4);
        // ---- joint-limit rows (btMultiBodyJointLimitConstraint): a lane owns at most one active row
        int lim_dir = 0; float lim_pen = 0.f;
        if (act && has_limit && alive) {
            float p0 = jp.x - LKo[kLLo], p1 = LKo[kLHi] - jp.x;
            if (!(p0 > 0.f)) { lim_dir = 1; lim_pen = p0; }
            else if (!(p1 > 0.f)) { lim_dir = -1; lim_pen = p1; }
        }
        const unsigned lbal = __ballot_sync(0xffffffffu, lim_dir != 0);
        const unsigned lseg = (W == 32) ? lbal : ((lbal >> (threadIdx.x & 16)) & 0xffffu);
        int NL = __popc(lseg);
        const unsigned anyrow = __ballot_sync(0xffffffffu, NL + P > 0);
        if (anyrow != 0) {
            {
                const int lidx = __popc(lseg & ((1u << lane) - 1u));
                if (NL > 8) { NL = 8; f_over = 1; }
                if (lim_dir != 0 && lidx < 8) { sQ[lidx] = __int_as_float(lane); sQ[8 + lidx] = (lim_dir == -1) ? -1.f : 1.f; sQ[16 + lidx] = lim_pen; sQ[24 + lidx] = jv.x; }
            }
            if (NL + 3 * P > LY.maxrows) { P = (LY.maxrows - NL) / 3; f_over = 1; }
            const int NR = NL + 3 * P;
            __syncwarp();
            PROF(5);
#ifdef DM_PROFILE
            { const int nrm = wmax(NR); if ((threadIdx.x & 31) == 0) { PRF[13] += nrm; PRF[14] += 1; if (nrm > W) PRF[15] += 1; } }
#endif
            solve_rows<W>(NL, P, mani, alive ? 1 : 0, PRFP);
            PROF(10);
            const float3 dq = dv_pass<W>();
            if (NR > 0) {
                if (ndof >= 1) jv.x = cl100(jv.x + dq.x);
                if (ndof == 3) { jv.y = cl100(jv.y + dq.y); jv.z = cl100(jv.z + dq.z); }
            }
            if (DEBUG && dbg && first_upd) {   // solver rows in solver order: right-hand side, 1 / A_ii, impulse (test hook)
                const float2* sRI_ = reinterpret_cast<const float2*>(E + LY.oRhs);
                for (int k = lane; k < NR && k < 64; k += W) { float* o = dbg + 8 * kMaxDofs + sub * 256; o[k] = sRI_[k].x; o[64 + k] = sRI_[k].y; o[128 + k] = sLam[k]; }
            }
            if (DEBUG && dbg && first_upd) {   // impulses in the order [normals | friction pairs | limits]
                const int lo_ = (sub == 0 ? 7 * kMaxDofs : 11 * kMaxDofs + 1024) + 1;
                for (int k = lane; k < NR && k < 60; k += W) { const int src = (k < 3 * P) ? NL + k : k - 3 * P; dbg[lo_ + k] = sLam[src]; }
            }
            PROF(11);
        }
        if (DEBUG && dbg && first_upd) {
            const int o = (sub == 0 ? 6 * kMaxDofs : 10 * kMaxDofs + 1024);
            if (lane == 0) for (int k = 0; k < 6; ++k) dbg[o + k] = sB[7 + k];
            if (ndof >= 1) dbg[o + dof0] = jv.x;
            if (ndof == 3) { dbg[o + dof0 + 1] = jv.y; dbg[o + dof0 + 2] = jv.z; }
        }
        // ---- integrate positions (btMultiBody::stepPositionsMultiDof)
        if (lane == 0) {
            sB[0] += h * sB[10]; sB[1] += h * sB[11]; sB[2] += h * sB[12];
            const Q4 q = quat_integrate3(mk3(sB[7], sB[8], sB[9]), mkq(sB[3], sB[4], sB[5], sB[6]), true, h);
            sB[3] = q.x; sB[4] = q.y; sB[5] = q.z; sB[6] = q.w;
        }
        if (jtype == kJRevolute) jp.x += h * jv.x;
        else if (jtype == kJSpherical) { Q4 q = quat_integrate3(mk3(jv.x, jv.y, jv.z), mkq(jp.x, jp.y, jp.z, jp.w), false, h); jp = make_float4(q.x, q.y, q.z, q.w); }
        __syncwarp();
        need_kin = true;
        if (ph == sim_substeps) pending_flags = true;
        PROF(12);
    }
#ifdef DM_PROFILE
    __syncwarp();
    if ((threadIdx.x & 31) == 0 && st.pdbg) { unsigned int* o = reinterpret_cast<unsigned int*>(st.pdbg) + (blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32) * 16; for (int k = 0; k < 16; ++k) o[k] = PRF[k]; }
#endif
}

// explicit instantiations used by capi.cu: (tile width, debug dumps)
template __global__ void dm_step_kernel<16, false, 0>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
template __global__ void dm_step_kernel<32, false, 0>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
template __global__ void dm_step_kernel<16, true, 0>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
template __global__ void dm_step_kernel<32, true, 0>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
// AMP task scenes (target_amp / heading_amp): same step with the task block advanced after every update
template __global__ void dm_step_kernel<16, false, kVarTask>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
template __global__ void dm_step_kernel<32, false, kVarTask>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
// --sync_char_root_rot true (dog3d_spin)
template __global__ void dm_step_kernel<16, false, kVarRootRot>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);
template __global__ void dm_step_kernel<32, false, kVarRootRot>(const DevModel*, DevState, const double*, const float*, double, int, int, StepLayout);

}  // namespace dmk
