// nb2_collide.cu - fused per-environment collision pipeline for sm_100a.
//
// One sub-warp group of L lanes owns one environment (a CTA is a single warp holding 32/L environments, so every
// synchronisation is a __syncwarp and ~14 independent CTAs per SM cover 4096 environments on 148 SMs in one wave):
//
//   phase 1  shape world transforms + AABBs          (reference sim/collide.py:283-472 compute_shape_aabbs)
//   phase 2  explicit-pair AABB test                 (reference geometry/broad_phase_nxn.py:29-69)
//            analytic narrow phase                   (reference geometry/narrow_phase.py:459-1014,
//                                                     geometry/collision_primitive.py)
//            GJK/MPR + manifold for convex pairs     (reference geometry/narrow_phase.py:1041-1216)   [nb2_gjk.cuh]
//            contact write-out                       (reference sim/collide.py:166-254 write_contact)
//
// The candidate-pair queue, the global atomic slot counter and the GJK re-queue of the reference disappear: the
// env's pair list is pre-sorted by the deterministic contact key, so a segmented prefix sum inside the group gives
// every contact its slot in key order - the order `CollisionPipeline(deterministic=True)` produces by radix sort.
// Contacts land in env-major SoA "contact blocks" that the solver kernels read directly; an optional export pass
// (scan + scatter) compacts them into the reference `Contacts` arrays.
#include <cub/device/device_radix_sort.cuh>

#include "nb2_gjk.cuh"

#include "nb2_internal.cuh"
#include "nb2_math.cuh"

namespace nb2 {

enum { GEO_PLANE = 1, GEO_SPHERE = 3, GEO_CAPSULE = 4, GEO_ELLIPSOID = 5, GEO_CYLINDER = 6, GEO_BOX = 7, GEO_MESH = 8, GEO_CONE = 9, GEO_CONVEX_MESH = 10 };
#define NB2_MAXVAL 1.0e10f

// ---- analytic colliders --------------------------------------------------------------------------
NB2_DEV void plane_sphere(V3 n, V3 pp, V3 sp, float r, float& dist, V3& pos) {
    dist = dot(sp - pp, n) - r;
    pos = sp - n * (r + 0.5f * dist);
}
NB2_DEV void sphere_sphere(V3 p1, float r1, V3 p2, float r2, float& dist, V3& pos, V3& n) {
    V3 dir = p2 - p1;
    float d = len(dir);
    n = d == 0.0f ? V3(1.f, 0.f, 0.f) : dir / d;
    dist = d - (r1 + r2);
    pos = p1 + n * (r1 + 0.5f * dist);
}
NB2_DEV V3 closest_on_segment(V3 a, V3 b, V3 pt) {
    V3 ab = b - a;
    float t = dot(pt - a, ab) / (dot(ab, ab) + 1e-6f);
    return a + clamp_w(t, 0.0f, 1.0f) * ab;
}
NB2_DEV void plane_box(V3 n, V3 pp, V3 bp, const M33& R, V3 half, float margin, float dist[4], V3 pos[4]) {
    float center_dist = dot(bp - pp, n);
    int ncontact = 0, worst = 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        V3 c((i & 1) ? half.x : -half.x, (i & 2) ? half.y : -half.y, (i & 4) ? half.z : -half.z);
        c = mv(R, c);
        float cdist = center_dist + dot(n, c);
        if (cdist > margin) continue;
        V3 cpos = c + bp - 0.5f * n * cdist;
        if (ncontact < 4) {
            dist[ncontact] = cdist;
            pos[ncontact] = cpos;
            if (ncontact == 0 || cdist > dist[worst]) worst = ncontact;
            ncontact += 1;
        } else if (cdist < dist[worst]) {
            dist[worst] = cdist;
            pos[worst] = cpos;
            worst = 0;
            if (dist[1] > dist[worst]) worst = 1;
            if (dist[2] > dist[worst]) worst = 2;
            if (dist[3] > dist[worst]) worst = 3;
        }
    }
}
NB2_DEV void plane_cylinder(V3 n, V3 pp, V3 cp, V3 axis, float radius, float hh, float dist[4], V3 pos[4]) {
    const float kFlatCos = 0.92387953251128673848f;  // cos 22.5 deg
    float dna = dot(n, axis);
    if (dna > 0.0f) {
        axis = -axis;
        dna = -dna;
    }
    V3 cap = cp + axis * hh;
    V3 perp_align = -n + axis * dna;
    float pl2 = dot(perp_align, perp_align);
    bool has_align = pl2 > 1e-10f;
    if (has_align) perp_align = perp_align * (1.0f / sqrtf(pl2));
    bool flat = (-dna) >= kFlatCos;
    V3 perp_fixed;
    if (flat || !has_align) {
        V3 ref(1.f, 0.f, 0.f);
        if (fabsf(dot(axis, ref)) > 0.9f) ref = V3(0.f, 1.f, 0.f);
        perp_fixed = unit(ref - axis * dot(axis, ref));
    }
    V3 deepest_perp = has_align ? perp_align : perp_fixed;
    V3 dpt = cap + deepest_perp * radius;
    float dd = dot(dpt - pp, n);
    V3 dpos = dpt - n * (dd * 0.5f);
    dist[0] = dd;
    pos[0] = dpos;
    int nc = 1;
    float mt = 0.01f * fmax_w(radius, hh);
    float mt2 = mt * mt;
    if (flat) {
        V3 u = perp_fixed * radius;
        V3 v = cross(axis, perp_fixed) * radius;
        const float c120 = -0.5f, s120 = 0.8660254f;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            V3 pt = k == 0 ? cap + u : (k == 1 ? cap + c120 * u + s120 * v : cap + c120 * u - s120 * v);
            float d = dot(pt - pp, n);
            V3 p = pt - n * (d * 0.5f);
            if (nc < 4 && len2(p - dpos) > mt2) {
                dist[nc] = d;
                pos[nc] = p;
                nc += 1;
            }
        }
    } else {
        V3 perp_roll = has_align ? perp_align : perp_fixed;
        V3 u = perp_roll * radius;
        V3 v = cross(axis, perp_roll) * radius;
        V3 pt = cp - axis * hh + u;
        float d = dot(pt - pp, n);
        V3 p = pt - n * (d * 0.5f);
        if (nc < 4 && len2(p - dpos) > mt2) {
            dist[nc] = d;
            pos[nc] = p;
            nc += 1;
        }
        V3 ptp = cap + v, ptn = cap - v;
        float dp = dot(ptp - pp, n), dn = dot(ptn - pp, n);
        bool use_p = dp <= dn;
        pt = use_p ? ptp : ptn;
        d = use_p ? dp : dn;
        p = pt - n * (d * 0.5f);
        if (nc < 4 && len2(p - dpos) > mt2) {
            dist[nc] = d;
            pos[nc] = p;
            nc += 1;
        }
    }
}
NB2_DEV void capsule_capsule(V3 p1, V3 a1, float r1, float hl1, V3 p2, V3 a2, float r2, float hl2, float dist[4], V3 pos[4], V3& n) {
    V3 ax1 = a1 * hl1, ax2 = a2 * hl2, dif = p1 - p2;
    float ma = dot(ax1, ax1), mb = -dot(ax1, ax2), mc = dot(ax2, ax2), u = -dot(ax1, dif), v = dot(ax2, dif);
    float det = ma * mc - mb * mb;
    if (fabsf(det) >= 1e-15f) {
        float inv_det = 1.0f / det;
        float x1 = (mc * u - mb * v) * inv_det, x2 = (ma * v - mb * u) * inv_det;
        if (x1 > 1.0f) { x1 = 1.0f; x2 = (v - mb) / mc; }
        else if (x1 < -1.0f) { x1 = -1.0f; x2 = (v + mb) / mc; }
        if (x2 > 1.0f) { x2 = 1.0f; x1 = clamp_w((u - mb) / ma, -1.0f, 1.0f); }
        else if (x2 < -1.0f) { x2 = -1.0f; x1 = clamp_w((u + mb) / ma, -1.0f, 1.0f); }
        sphere_sphere(p1 + ax1 * x1, r1, p2 + ax2 * x2, r2, dist[0], pos[0], n);
    } else {
        float x2 = clamp_w((v - mb) / mc, -1.0f, 1.0f);
        sphere_sphere(p1 + ax1, r1, p2 + ax2 * x2, r2, dist[0], pos[0], n);
        x2 = clamp_w((v + mb) / mc, -1.0f, 1.0f);
        V3 n2;
        sphere_sphere(p1 - ax1, r1, p2 + ax2 * x2, r2, dist[1], pos[1], n2);
    }
}
NB2_DEV void sphere_cylinder(V3 sp, float sr, V3 cp, V3 axis, float cr, float chh, float& dist, V3& pos, V3& n) {
    V3 vec = sp - cp;
    float x = dot(vec, axis);
    V3 a_proj = axis * x;
    V3 p_proj = vec - a_proj;
    float pp2 = dot(p_proj, p_proj);
    bool side = fabsf(x) < chh, capc = pp2 < cr * cr;
    if (side && capc) {
        float dist_cap = chh - fabsf(x), dist_radius = cr - sqrtf(pp2);
        if (dist_cap < dist_radius) side = false;
        else capc = false;
    }
    if (side) {
        sphere_sphere(sp, sr, cp + a_proj, cr, dist, pos, n);
    } else if (capc) {
        V3 pc, pn;
        if (x > 0.0f) { pc = cp + axis * chh; pn = axis; }
        else { pc = cp - axis * chh; pn = -axis; }
        plane_sphere(pn, pc, sp, sr, dist, pos);
        n = -pn;
    } else {
        float s = sqrtf(pp2);
        float inv_len = 1.0f / (s != 0.0f ? s : 1e-15f);
        p_proj = p_proj * (cr * inv_len);
        V3 cap_offset = axis * ((x < 0.0f ? -1.0f : 1.0f) * chh);
        sphere_sphere(sp, sr, cp + cap_offset + p_proj, 0.0f, dist, pos, n);
    }
}
NB2_DEV void sphere_box(V3 sp, float sr, V3 bp, const M33& R, V3 half, float& dist, V3& position, V3& n) {
    V3 center = mtv(R, sp - bp);
    V3 clamped = vmax(-half, vmin(half, center));
    V3 diff = clamped - center;
    float d = len(diff);
    V3 dir = d == 0.0f ? diff : diff / d;
    V3 pos;
    if (d <= 1e-6f) {
        float closest = 2.0f * (half.x + half.y + half.z);
        int k = 0;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            float fd = fabsf(((i % 2) ? 1.0f : -1.0f) * half.get(i / 2) - center.get(i / 2));
            if (closest > fd) { closest = fd; k = i; }
        }
        V3 nearest;
        nearest.set(k / 2, (k % 2) ? -1.0f : 1.0f);
        pos = center + nearest * (sr - closest) / 2.0f;
        n = mv(R, nearest);
        dist = -closest - sr;
    } else {
        V3 deepest = center + dir * sr;
        pos = 0.5f * (clamped + deepest);
        n = mv(R, dir);
        dist = d - sr;
    }
    position = bp + mv(R, pos);
}

// World AABB of one shape, expanded by margin + gap (compute_shape_aabbs).
NB2_DEV void shape_aabb(int type, V3 scale, const Xf& X, float gap_eff, float coll_radius, V3 local_lo, V3 local_hi, V3& lo, V3& hi) {
    V3 pos = X.p;
    V3 mvv(gap_eff, gap_eff, gap_eff);
    V3 he;
    if (type == GEO_CONVEX_MESH || type == GEO_MESH) {  // has_local_aabb (collide.py:348, 420-444): the builder's scaled local AABB rotated into the world
        const V3 center = (local_lo + local_hi) * 0.5f, half = (local_hi - local_lo) * 0.5f;
        const V3 wc = qrot(X.q, center) + pos;
        const V3 r0 = qrot(X.q, V3(1.f, 0.f, 0.f)), r1 = qrot(X.q, V3(0.f, 1.f, 0.f)), r2 = qrot(X.q, V3(0.f, 0.f, 1.f));
        const V3 wh(fabsf(r0.x) * half.x + fabsf(r1.x) * half.y + fabsf(r2.x) * half.z,
                    fabsf(r0.y) * half.x + fabsf(r1.y) * half.y + fabsf(r2.y) * half.z,
                    fabsf(r0.z) * half.x + fabsf(r1.z) * half.y + fabsf(r2.z) * half.z);
        lo = wc - wh - mvv;
        hi = wc + wh + mvv;
        return;
    }
    if (type == GEO_PLANE && scale.x == 0.0f && scale.y == 0.0f) {
        V3 normal = qrot(X.q, V3(0.f, 0.f, 1.f));
        const float EXT = 1.0e6f;
        V3 e(EXT, EXT, EXT);
        lo = pos - e - mvv;
        hi = pos + e + mvv;
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            float ni = normal.get(i);
            if (fabsf(ni) > 0.5f) {
                float lateral = fabsf(normal.get((i + 1) % 3)) + fabsf(normal.get((i + 2) % 3));
                float rise = lateral * EXT / fabsf(ni);
                if (ni > 0.0f) hi.set(i, fmin_w(hi.get(i), pos.get(i) + rise + gap_eff));
                else lo.set(i, fmax_w(lo.get(i), pos.get(i) - rise - gap_eff));
            }
        }
        return;
    } else if (type == GEO_SPHERE) {
        he = V3(scale.x, scale.x, scale.x);
    } else if (type == GEO_BOX) {
        V3 r0 = qrot(X.q, V3(1.f, 0.f, 0.f)), r1 = qrot(X.q, V3(0.f, 1.f, 0.f)), r2 = qrot(X.q, V3(0.f, 0.f, 1.f));
        he = V3(fabsf(r0.x) * scale.x + fabsf(r1.x) * scale.y + fabsf(r2.x) * scale.z,
                fabsf(r0.y) * scale.x + fabsf(r1.y) * scale.y + fabsf(r2.y) * scale.z,
                fabsf(r0.z) * scale.x + fabsf(r1.z) * scale.y + fabsf(r2.z) * scale.z);
    } else if (type == GEO_CAPSULE) {
        V3 axis = qrot(X.q, V3(0.f, 0.f, 1.f));
        he = V3(scale.x, scale.x, scale.x) + vabs(axis) * scale.y;
    } else if (type == GEO_CYLINDER) {
        float radius = scale.x, hh = scale.y, br = scale.z;
        if (br >= hh && br > 0.0f) radius += (hh * hh) / (br + sqrtf(br * br - hh * hh));
        V3 r0 = qrot(X.q, V3(1.f, 0.f, 0.f)), r1 = qrot(X.q, V3(0.f, 1.f, 0.f)), r2 = qrot(X.q, V3(0.f, 0.f, 1.f));
        he = V3(radius * sqrtf(r0.x * r0.x + r1.x * r1.x) + hh * fabsf(r2.x), radius * sqrtf(r0.y * r0.y + r1.y * r1.y) + hh * fabsf(r2.y),
                radius * sqrtf(r0.z * r0.z + r1.z * r1.z) + hh * fabsf(r2.z));
    } else if (type == GEO_CONE || type == GEO_PLANE) {  // generic branch of compute_shape_aabbs: tight AABB from the support map
        // (finite planes: geom_scale holds HALF extents, collide.py:452-453)
        const ConvexGeom g{type, type == GEO_PLANE ? V3(scale.x * 0.5f, scale.y * 0.5f, 0.0f) : scale};
        tight_aabb_from_support(g, X.q, pos, lo, hi);
        lo = lo - mvv;
        hi = hi + mvv;
        return;
    } else if (type == GEO_ELLIPSOID) {
        M33 R = qmat(X.q);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            float a = R.at(i, 0) * scale.x, b = R.at(i, 1) * scale.y, c = R.at(i, 2) * scale.z;
            he.set(i, sqrtf(a * a + b * b + c * c));
        }
    } else {
        he = V3(coll_radius, coll_radius, coll_radius);
    }
    lo = pos - he - mvv;
    hi = pos + he + mvv;
}

// compute_shape_velocities (sim/collide.py:475-541) for one shape whose world transform X_ws is known: shape-origin velocity,
// angular velocity, velocity-extended search gap, displacement over the collision-update interval; the AABB grows by the (capped)
// angular travel.  Static shapes (body -1) keep zero motion and their authored gap.
struct ShapeMotion {
    V3 lin, ang, disp;
    float search_gap;
};
NB2_DEV ShapeMotion shape_motion(const DevModel& M, const float* __restrict__ body_q, int sid, int body, const Xf& X_ws, V3& lo, V3& hi) {
    const nb2_model_desc& d = M.d;
    ShapeMotion o;
    o.search_gap = d.shape_gap[sid];
    if (body == -1) return o;
    const Xf X_wb = ldx(body_q + 7 * body);
    const V3 com_world = xpoint(X_wb, ld3(d.body_com + 3 * body));
    const V3 com_velocity = ld3(M.spec_body_qd + 6 * body), angular_velocity = ld3(M.spec_body_qd + 6 * body + 3);
    const V3 origin_velocity = com_velocity + cross(angular_velocity, X_ws.p - com_world);
    o.lin = origin_velocity;
    o.ang = angular_velocity;
    const V3 furthest = vmax(vabs(ld3(d.shape_collision_aabb_lower + 3 * sid)), vabs(ld3(d.shape_collision_aabb_upper + 3 * sid)));
    const float angular_radius = fmax_w(len(furthest), d.shape_collision_radius[sid]);
    const float angular_speed_bound = len(angular_velocity) * angular_radius;
    const float search_extension = fmin_w((len(origin_velocity) + angular_speed_bound) * M.spec_dt, M.spec_max_ext);
    o.search_gap = d.shape_gap[sid] + search_extension;
    o.disp = origin_velocity * M.spec_dt;
    const float ae = fmin_w(angular_speed_bound * M.spec_dt, M.spec_max_ext);
    lo = lo - V3(ae, ae, ae);
    hi = hi + V3(ae, ae, ae);
    return o;
}
// check_aabb_overlap_moving (broad_phase_common.py:41-80, cutoffs 0): box 1 swept by the RELATIVE displacement against box 2
NB2_DEV bool aabb_overlap_moving(V3 lo1, V3 hi1, V3 lo2, V3 hi2, V3 rel) {
    float enter = 0.0f, exit_time = 1.0f;
#pragma unroll
    for (int axis = 0; axis < 3; ++axis) {
        const float lower1 = lo1.get(axis), upper1 = hi1.get(axis), lower2 = lo2.get(axis), upper2 = hi2.get(axis), delta = rel.get(axis);
        if (delta == 0.0f) {
            if (lower1 > upper2 || upper1 < lower2) return false;
        } else {
            float axis_enter = (lower2 - upper1) / delta, axis_exit = (upper2 - lower1) / delta;
            if (axis_enter > axis_exit) {
                const float t = axis_enter;
                axis_enter = axis_exit;
                axis_exit = t;
            }
            enter = fmax_w(enter, axis_enter);
            exit_time = fmin_w(exit_time, axis_exit);
            if (enter > exit_time) return false;
        }
    }
    return true;
}
// prepare_speculative_contact + contact_passes_speculative_gap_check (contact_data.py:187-233)
NB2_DEV bool speculative_admit(const ShapeMotion& ma, V3 origin_a, const ShapeMotion& mb, V3 origin_b, V3 center, V3 nn, float dist, float reff_a,
                               float reff_b, float total_sep, float base_gap_sum, float dt, float max_ext) {
    const V3 a_w = center - nn * (0.5f * dist + reff_a);
    const V3 b_w = center + nn * (0.5f * dist + reff_b);
    const float separation = dot(b_w - a_w, nn) - total_sep;
    if (separation <= base_gap_sum) return true;
    const V3 va = ma.lin + cross(ma.ang, a_w - origin_a), vb = mb.lin + cross(mb.ang, b_w - origin_b);
    const float approach = fmax_w(-dot(vb - va, nn), 0.0f);
    const float extension = fmin_w(approach * dt, max_ext);
    return extension - separation >= 0.0f;
}

struct PairGeom {
    int type;
    V3 scale;
    float margin, gap, radius;
    Xf X;
};

// Shared-memory record of one shape slot: world transform + expanded AABB.
struct __align__(4) SlotRec {
    float x[7];
    float lo[3];
    float hi[3];
};

// Write-out staging: the narrow phase leaves a pair's candidates in the registers of ONE lane - the 4
// contacts of a foot would be converted and stored by that lane one after the other while the group's other lanes idle.  Instead
// every lane drops its admitted candidates (and the pair's constants) into shared memory, and the group converts / stores them one
// lane per CONTACT: the write_contact code runs once per round instead of up to five times, and exists once in the binary.
// Measured against the one-lane-per-pair write-out: 656.1 -> 644.4 us per 4096-quadruped frame (profiles/r2l_min_grid_ab.txt).
struct __align__(4) StageContact {
    float center[3], normal[3], dist;
    int pair_lane;
};
struct __align__(4) StagePair {
    int sa, sb;
    float reff_a, reff_b, marg_a, marg_b;
};
__host__ __device__ inline size_t stage_bytes_per_group(int L) { return size_t(L) * 5 * sizeof(StageContact) + size_t(L) * sizeof(StagePair); }

// Speculative contacts only (DevModel::spec_mode != 0): per-slot motion record next to the SlotRec table
struct __align__(4) SlotMotionRec {
    float lin[3], ang[3], disp[3], search_gap;
};
NB2_DEV ShapeMotion ld_motion(const SlotMotionRec& r) {
    ShapeMotion o;
    o.lin = ld3(r.lin);
    o.ang = ld3(r.ang);
    o.disp = ld3(r.disp);
    o.search_gap = r.search_gap;
    return o;
}

// CONVEX = false is instantiated for models none of whose pairs can reach the generic convex path (decided per pair type at
// nb2_model_create): the analytic-only kernel carries neither the MPR / GJK / manifold code nor its registers and stack.
// WARPS warps per CTA (each warp = 32/L environments): the kernel is a straight line every warp walks once, so one-warp CTAs each
// fetch the whole instruction stream cold (48 % `stall_no_inst`, profiles/r1f_collide_kernel_quadruped.txt); warps of one CTA
// start together and share the fetches.
template <int L, bool CONVEX, int WARPS>
__global__ void __launch_bounds__(32 * WARPS) collide_kernel(DevModel M, const float* __restrict__ body_q) {
    constexpr int G = 32 / L;  // environments per warp
    extern __shared__ unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / L;
    const int l = lane % L;
    const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << (grp * L));
    const int env = (blockIdx.x * WARPS + warp) * G + grp;
    const bool live = env < M.env_count;
    SlotRec* slots = reinterpret_cast<SlotRec*>(smem_raw) + size_t(warp * G + grp) * M.max_env_slots_shapes;
    const nb2_model_desc& d = M.d;
    // speculative contacts run in the generic instantiation only (launch_collide picks CONVEX = true for them)
    const int spec_mode = CONVEX ? M.spec_mode : 0;
    SlotMotionRec* motion = nullptr;
    if (CONVEX && spec_mode != 0)
        motion = reinterpret_cast<SlotMotionRec*>(reinterpret_cast<SlotRec*>(smem_raw) + size_t(WARPS * G) * M.max_env_slots_shapes) +
                 size_t(warp * G + grp) * M.max_env_slots_shapes;
    unsigned char* sbase = smem_raw + size_t(WARPS * G) * M.max_env_slots_shapes * (sizeof(SlotRec) + (CONVEX && spec_mode != 0 ? sizeof(SlotMotionRec) : 0)) +
                           size_t(warp * G + grp) * stage_bytes_per_group(L);
    StageContact* stage_c = reinterpret_cast<StageContact*>(sbase);
    StagePair* stage_p = reinterpret_cast<StagePair*>(sbase + size_t(L) * 5 * sizeof(StageContact));

    int ss = 0, nloc = 0, nslots = 0, bs = 0, ps = 0, np = 0, slot0 = 0;
    if (live) {
        ss = M.env_shape_start[env];
        nloc = M.env_shape_start[env + 1] - ss;
        nslots = nloc + M.global_shape_count;
        bs = M.env_body_start[env];
        if (M.dyn_pairs) {  // run-time broad phase: the candidates broadphase_kernel left for this env
            ps = env * M.dyn_pair_cap;
            np = min(M.env_dyn_count[env], M.dyn_pair_cap);
        } else {
            ps = M.env_pair_start[env];
            np = M.env_pair_start[env + 1] - ps;
        }
        slot0 = M.env_slot_start[env];
    }
    // ---- phase 1: transforms + AABBs -----------------------------------------------------------
    for (int s = l; s < nslots; s += L) {
        int sid = s < nloc ? ss + s : M.global_shapes[s - nloc];
        int body = d.shape_body[sid];
        Xf X = ldx(d.shape_transform + 7 * sid);
        if (body != -1) X = xmul(ldx(body_q + 7 * body), X);
        float margin = d.shape_margin[sid];
        V3 lo, hi;
        const int stype = d.shape_type[sid];
        V3 llo, lhi;
        if (stype == GEO_CONVEX_MESH || stype == GEO_MESH) {
            llo = ld3(d.shape_collision_aabb_lower + 3 * sid);
            lhi = ld3(d.shape_collision_aabb_upper + 3 * sid);
        }
        shape_aabb(stype, ld3(d.shape_scale + 3 * sid), X, margin + d.shape_gap[sid], d.shape_collision_radius[sid], llo, lhi, lo, hi);
        if (CONVEX && motion) {
            ShapeMotion mo;
            mo.search_gap = d.shape_gap[sid];
            if (spec_mode == 2) mo = shape_motion(M, body_q, sid, body, X, lo, hi);
            st3(motion[s].lin, mo.lin);
            st3(motion[s].ang, mo.ang);
            st3(motion[s].disp, mo.disp);
            motion[s].search_gap = mo.search_gap;
        }
        stx(slots[s].x, X);
        st3(slots[s].lo, lo);
        st3(slots[s].hi, hi);
    }
    __syncwarp();
    if (WARPS > 1) __syncthreads();  // alignment only (see above)
    // ---- phase 2: pairs -> contacts -------------------------------------------------------------
    int n_total = 0;
    const int rounds = (np + L - 1) / L;
    int max_rounds = rounds;
#pragma unroll
    for (int o = 16; o >= L; o >>= 1) max_rounds = max(max_rounds, __shfl_xor_sync(0xffffffffu, max_rounds, o));
    for (int r = 0; r < max_rounds; ++r) {
        const int p = r * L + l;
        unsigned vmask = 0;  // bit i set -> contact candidate i of this pair is emitted
        float cdist[5];
        V3 cpos[5], cnorm[5];
        int sa = 0, sb = 0;
        float reff_a = 0.f, reff_b = 0.f, marg_a = 0.f, marg_b = 0.f;
        int mesh_a = -1, mesh_b = -1;  // slots of an overlapping (mesh, infinite plane) pair: handled by the whole group below
        if (live && p < np) {
            int2 pr = M.dyn_pairs ? M.dyn_pairs[ps + p] : M.pairs[ps + p];
            const bool mesh_pair = CONVEX && (pr.y & NB2_PAIR_MESH_PLANE) != 0;  // explicit list only (nb2_model_create)
            pr.y &= ~NB2_PAIR_MESH_PLANE;
            V3 alo = ld3(slots[pr.x].lo), ahi = ld3(slots[pr.x].hi), blo = ld3(slots[pr.y].lo), bhi = ld3(slots[pr.y].hi);
            bool overlap = alo.x <= bhi.x && ahi.x >= blo.x && alo.y <= bhi.y && ahi.y >= blo.y && alo.z <= bhi.z && ahi.z >= blo.z;
            if (CONVEX && spec_mode == 2)  // swept test over the relative displacement (the explicit sweep passes (s1, s2) = the stored pair)
                overlap = aabb_overlap_moving(alo, ahi, blo, bhi, ld3(motion[pr.x].disp) - ld3(motion[pr.y].disp));
            if (overlap && !M.include_static_kinematic_pairs && !M.dyn_pairs) {
                // is_shape_pair_immovable_filtered (broad_phase_common.py:166-201) in the explicit sweep (broad_phase_nxn.py:29-69)
                const int s1 = pr.x < nloc ? ss + pr.x : M.global_shapes[pr.x - nloc], s2 = pr.y < nloc ? ss + pr.y : M.global_shapes[pr.y - nloc];
                const int b1 = d.shape_body[s1], b2 = d.shape_body[s2];
                const bool im1 = b1 < 0 || (d.body_flags[b1] & 2) != 0, im2 = b2 < 0 || (d.body_flags[b2] & 2) != 0;
                if (im1 && im2) overlap = false;
            }
            if (CONVEX && overlap && mesh_pair) {
                mesh_a = pr.x;
                mesh_b = pr.y;
                overlap = false;
            }
            if (overlap) {
                sa = pr.x < nloc ? ss + pr.x : M.global_shapes[pr.x - nloc];
                sb = pr.y < nloc ? ss + pr.y : M.global_shapes[pr.y - nloc];
                const int ta = d.shape_type[sa], tb = d.shape_type[sb];
                V3 sca = ld3(d.shape_scale + 3 * sa), scb = ld3(d.shape_scale + 3 * sb);
                Xf Xa = ldx(slots[pr.x].x), Xb = ldx(slots[pr.y].x);
                marg_a = d.shape_margin[sa];
                marg_b = d.shape_margin[sb];
                // speculative: the colliders see the velocity-extended search gaps, the admission test the authored ones
                const float base_gap_sum = d.shape_gap[sa] + d.shape_gap[sb];
                const float gap_sum = (CONVEX && spec_mode == 2) ? motion[pr.x].search_gap + motion[pr.y].search_gap : base_gap_sum;
                const bool early_gjk = ta >= GEO_ELLIPSOID || tb == GEO_CONE || (ta == GEO_CAPSULE && tb > GEO_CAPSULE);
                bool analytic = false;
                float dist[4] = {NB2_MAXVAL, NB2_MAXVAL, NB2_MAXVAL, NB2_MAXVAL};
                V3 pos[4], normal;
                if (!early_gjk) {
                    if (ta == GEO_SPHERE || ta == GEO_CAPSULE) reff_a = sca.x;
                    if (tb == GEO_SPHERE || tb == GEO_CAPSULE) reff_b = scb.x;
                    analytic = true;
                    bool use_pc = ta == GEO_PLANE && tb == GEO_CYLINDER;
                    if (use_pc && scb.z > 0.0f) {
                        V3 pn = qrot(Xa.q, V3(0.f, 0.f, 1.f)), ca = qrot(Xb.q, V3(0.f, 0.f, 1.f));
                        use_pc = fabsf(dot(pn, ca)) * scb.z >= scb.y;
                    }
                    if (ta == GEO_PLANE && tb == GEO_SPHERE) {
                        normal = qrot(Xa.q, V3(0.f, 0.f, 1.f));
                        plane_sphere(normal, Xa.p, Xb.p, scb.x, dist[0], pos[0]);
                    } else if (ta == GEO_PLANE && tb == GEO_ELLIPSOID) {
                        V3 pn = qrot(Xa.q, V3(0.f, 0.f, 1.f));
                        M33 R = qmat(Xb.q);
                        V3 sup = -unit(cmul(mtv(R, pn), scb));
                        V3 pt = Xb.p + mv(R, cmul(sup, scb));
                        dist[0] = dot(pn, pt - Xa.p);
                        pos[0] = pt - pn * dist[0] * 0.5f;
                        normal = pn;
                    } else if (ta == GEO_PLANE && tb == GEO_BOX) {
                        normal = qrot(Xa.q, V3(0.f, 0.f, 1.f));
                        plane_box(normal, Xa.p, Xb.p, qmat(Xb.q), scb, gap_sum + marg_a + marg_b, dist, pos);
                    } else if (ta == GEO_SPHERE && tb == GEO_SPHERE) {
                        sphere_sphere(Xa.p, sca.x, Xb.p, scb.x, dist[0], pos[0], normal);
                    } else if (ta == GEO_PLANE && tb == GEO_CAPSULE) {
                        normal = qrot(Xa.q, V3(0.f, 0.f, 1.f));
                        V3 seg = qrot(Xb.q, V3(0.f, 0.f, 1.f)) * scb.y;
                        plane_sphere(normal, Xa.p, Xb.p + seg, scb.x, dist[0], pos[0]);
                        plane_sphere(normal, Xa.p, Xb.p - seg, scb.x, dist[1], pos[1]);
                    } else if (use_pc) {
                        normal = qrot(Xa.q, V3(0.f, 0.f, 1.f));
                        plane_cylinder(normal, Xa.p, Xb.p, qrot(Xb.q, V3(0.f, 0.f, 1.f)), scb.x, scb.y, dist, pos);
                    } else if (ta == GEO_SPHERE && tb == GEO_CAPSULE) {
                        V3 seg = qrot(Xb.q, V3(0.f, 0.f, 1.f)) * scb.y;
                        V3 pt = closest_on_segment(Xb.p - seg, Xb.p + seg, Xa.p);
                        sphere_sphere(Xa.p, sca.x, pt, scb.x, dist[0], pos[0], normal);
                    } else if (ta == GEO_CAPSULE && tb == GEO_CAPSULE) {
                        capsule_capsule(Xa.p, qrot(Xa.q, V3(0.f, 0.f, 1.f)), sca.x, sca.y, Xb.p, qrot(Xb.q, V3(0.f, 0.f, 1.f)), scb.x,
                                        scb.y, dist, pos, normal);
                    } else if (ta == GEO_SPHERE && tb == GEO_CYLINDER && scb.z == 0.0f) {
                        sphere_cylinder(Xa.p, sca.x, Xb.p, qrot(Xb.q, V3(0.f, 0.f, 1.f)), scb.x, scb.y, dist[0], pos[0], normal);
                    } else if (ta == GEO_SPHERE && tb == GEO_BOX) {
                        sphere_box(Xa.p, sca.x, Xb.p, qmat(Xb.q), scb, dist[0], pos[0], normal);
                    } else {
                        analytic = false;
                    }
                }
                if (analytic) {
                    const float tsn = reff_a + reff_b + marg_a + marg_b;
                    const V3 nn = unit(normal);
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        cdist[i] = dist[i];
                        cpos[i] = pos[i];
                        cnorm[i] = normal;
                        if (dist[i] < NB2_MAXVAL) {
                            // _contact_passes_gap_check_precomputed (contact_data.py:138-156)
                            if (CONVEX && spec_mode != 0) {
                                if (speculative_admit(ld_motion(motion[pr.x]), Xa.p, ld_motion(motion[pr.y]), Xb.p, pos[i], nn, dist[i], reff_a, reff_b,
                                                      tsn, base_gap_sum, M.spec_dt, M.spec_max_ext))
                                    vmask |= 1u << i;
                                continue;
                            }
                            V3 a_w = pos[i] - nn * (0.5f * dist[i] + reff_a);
                            V3 b_w = pos[i] + nn * (0.5f * dist[i] + reff_b);
                            float dd = dot(b_w - a_w, nn) - tsn;
                            if (dd <= gap_sum) vmask |= 1u << i;
                        }
                    }
                } else if (CONVEX) {
                    ConvexShape A{ta, sca, Xa, marg_a, d.shape_gap[sa], alo, ahi};
                    ConvexShape Bc{tb, scb, Xb, marg_b, d.shape_gap[sb], blo, bhi};
                    ConvexSpec cs;
                    if (spec_mode != 0) {
                        const ShapeMotion ma = ld_motion(motion[pr.x]), mb = ld_motion(motion[pr.y]);
                        A.gap = ma.search_gap;  // == the authored gap when speculation is inactive
                        Bc.gap = mb.search_gap;
                        cs.base_gap_sum = base_gap_sum;
                        cs.dt = M.spec_dt;
                        cs.max_extension = M.spec_max_ext;
                        cs.origin_a = Xa.p;
                        cs.origin_b = Xb.p;
                        cs.lin_a = ma.lin;
                        cs.lin_b = mb.lin;
                        cs.ang_a = ma.ang;
                        cs.ang_b = mb.ang;
                    }
                    if (ta == GEO_CONVEX_MESH) {  // narrow_phase.py:1096-1105
                        A.hull = d.hull_points + 3 * size_t(d.shape_hull_start[sa]);
                        A.hull_count = d.shape_hull_count[sa];
                        A.center = 0.5f * (ld3(d.shape_collision_aabb_lower + 3 * sa) + ld3(d.shape_collision_aabb_upper + 3 * sa));
                    }
                    if (tb == GEO_CONVEX_MESH) {
                        Bc.hull = d.hull_points + 3 * size_t(d.shape_hull_start[sb]);
                        Bc.hull_count = d.shape_hull_count[sb];
                        Bc.center = 0.5f * (ld3(d.shape_collision_aabb_lower + 3 * sb) + ld3(d.shape_collision_aabb_upper + 3 * sb));
                    }
                    vmask = convex_pair_contacts(A, Bc, cdist, cpos, cnorm, reff_a, reff_b, spec_mode != 0 ? &cs : nullptr);
                }
            }
        }
        // A round's contacts leave in pair order.  A (mesh, plane) pair emits one contact per vertex - far more than a lane's five
        // candidates - so the round is cut into segments at the mesh lanes: [staged pairs][mesh pair k][staged pairs] ..., each written
        // behind the previous one.  Rounds without mesh pairs (every round of the analytic-only instantiation) are one segment.
        unsigned mesh_lanes = 0;
        int nseg = 1;
        if (CONVEX && M.has_mesh_pairs) {
            mesh_lanes = (__ballot_sync(0xffffffffu, mesh_a >= 0) >> (grp * L)) & (L == 32 ? 0xffffffffu : ((1u << L) - 1u));
            nseg = 1 + __popc(mesh_lanes);
#pragma unroll
            for (int o = 16; o >= L; o >>= 1) nseg = max(nseg, __shfl_xor_sync(0xffffffffu, nseg, o));  // warp-uniform trip count
        }
        int seg_lo = 0;
        for (int seg = 0; seg < nseg; ++seg) {
            const int seg_hi = mesh_lanes ? __ffs(mesh_lanes) - 1 : L;  // next mesh lane of this group, or the end of the round
            const int cnt = (l >= seg_lo && l < seg_hi) ? __popc(vmask) : 0;
            // segmented exclusive scan of cnt over the L lanes of this group
            int incl = cnt;
    #pragma unroll
            for (int o = 1; o < L; o <<= 1) {
                int v = __shfl_up_sync(0xffffffffu, incl, o, L);
                if (l >= o) incl += v;
            }
            const int total = __shfl_sync(0xffffffffu, incl, L - 1, L);
            if (cnt > 0) {
                StagePair& sp = stage_p[l];
                sp.sa = sa; sp.sb = sb;
                sp.reff_a = reff_a; sp.reff_b = reff_b; sp.marg_a = marg_a; sp.marg_b = marg_b;
                int k = incl - cnt;
    #pragma unroll
                for (int i = 0; i < 5; ++i) {
                    if (!(vmask & (1u << i))) continue;
                    StageContact& sc = stage_c[k++];
                    st3(sc.center, cpos[i]);
                    st3(sc.normal, cnorm[i]);
                    sc.dist = cdist[i];
                    sc.pair_lane = l;
                }
            }
            __syncwarp();
            float* cb = M.cb;
            const size_t T = size_t(M.slot_total);
            for (int c = l; c < total; c += L) {
                const StageContact& sc = stage_c[c];
                const StagePair& sp = stage_p[sc.pair_lane];
                const int psa = sp.sa, psb = sp.sb;
                const float ra = sp.reff_a, rb = sp.reff_b;
                const int body0 = d.shape_body[psa], body1 = d.shape_body[psb];
                const Xf Xbw_a = body0 == -1 ? Xf() : xinv(ldx(body_q + 7 * body0));
                const Xf Xbw_b = body1 == -1 ? Xf() : xinv(ldx(body_q + 7 * body1));
                const int o = slot0 + n_total + c;
                // write_contact (collide.py:210-254): world contact -> body-frame points / offsets
                const V3 n = unit(ld3(sc.normal)), center = ld3(sc.center);
                const V3 a_w = center - n * (0.5f * sc.dist + ra);
                const V3 b_w = center + n * (0.5f * sc.dist + rb);
                const float om_a = ra + sp.marg_a, om_b = rb + sp.marg_b;
                const V3 p0 = xpoint(Xbw_a, a_w), p1 = xpoint(Xbw_b, b_w);
                const V3 o0 = xvec(Xbw_a, om_a * n), o1 = xvec(Xbw_b, -om_b * n);
                cb[CF_BODY_A * T + o] = __int_as_float(body0 >= 0 ? body0 - bs : -1);
                cb[CF_BODY_B * T + o] = __int_as_float(body1 >= 0 ? body1 - bs : -1);
                cb[CF_SHAPE0 * T + o] = __int_as_float(psa);
                cb[CF_SHAPE1 * T + o] = __int_as_float(psb);
                cb[CF_P0X * T + o] = p0.x; cb[CF_P0Y * T + o] = p0.y; cb[CF_P0Z * T + o] = p0.z;
                cb[CF_P1X * T + o] = p1.x; cb[CF_P1Y * T + o] = p1.y; cb[CF_P1Z * T + o] = p1.z;
                cb[CF_O0X * T + o] = o0.x; cb[CF_O0Y * T + o] = o0.y; cb[CF_O0Z * T + o] = o0.z;
                cb[CF_O1X * T + o] = o1.x; cb[CF_O1Y * T + o] = o1.y; cb[CF_O1Z * T + o] = o1.z;
                cb[CF_NX * T + o] = n.x; cb[CF_NY * T + o] = n.y; cb[CF_NZ * T + o] = n.z;
                cb[CF_MARGIN0 * T + o] = om_a;
                cb[CF_MARGIN1 * T + o] = om_b;
                cb[CF_MU * T + o] = (d.shape_material_mu[psa] + d.shape_material_mu[psb]) / 2.0f;
                cb[CF_MU_TORSIONAL * T + o] = (d.shape_material_mu_torsional[psa] + d.shape_material_mu_torsional[psb]) / 2.0f;
                cb[CF_MU_ROLLING * T + o] = (d.shape_material_mu_rolling[psa] + d.shape_material_mu_rolling[psb]) / 2.0f;
                cb[CF_KE * T + o] = 0.5f * (d.shape_material_ke[psa] + d.shape_material_ke[psb]);
                cb[CF_KD * T + o] = 0.5f * (d.shape_material_kd[psa] + d.shape_material_kd[psb]);
                cb[CF_KF * T + o] = 0.5f * (d.shape_material_kf[psa] + d.shape_material_kf[psb]);
                cb[CF_KA * T + o] = 0.5f * (d.shape_material_ka[psa] + d.shape_material_ka[psb]);
            }
            __syncwarp();  // the staging area is rewritten in the next round
            n_total += total;
            if (CONVEX && seg_hi < L) {
                // ---- mesh vs infinite plane (narrow_phase.py:1761-1861, reduce_contacts=False): the group walks the vertices L at a
                // time; a vertex within gap + margin of the plane is a contact (shape_a = mesh, normal mesh -> plane), kept in vertex order
                const int ma = __shfl_sync(gmask, mesh_a, seg_hi, L), mb = __shfl_sync(gmask, mesh_b, seg_hi, L);
                const int msa = ma < nloc ? ss + ma : M.global_shapes[ma - nloc], psb = mb < nloc ? ss + mb : M.global_shapes[mb - nloc];
                const Xf Xm = ldx(slots[ma].x), Xp = ldx(slots[mb].x);
                const Xf Xp_inv = xinv(Xp);
                const V3 pn = xvec(Xp, V3(0.f, 0.f, 1.f));
                const V3 mscale = ld3(d.shape_scale + 3 * msa);
                const float marg_m = d.shape_margin[msa], marg_p = d.shape_margin[psb];
                const float gap_sum = d.shape_gap[msa] + d.shape_gap[psb];
                const float* verts = d.hull_points + 3 * size_t(d.shape_hull_start[msa]);
                const int nv = d.shape_hull_count[msa];
                const int body0 = d.shape_body[msa], body1 = d.shape_body[psb];
                const Xf Xbw_a = body0 == -1 ? Xf() : xinv(ldx(body_q + 7 * body0));
                const Xf Xbw_b = body1 == -1 ? Xf() : xinv(ldx(body_q + 7 * body1));
                int written = 0;
                for (int v0 = 0; v0 < nv; v0 += L) {
                    const int vi = v0 + l;
                    bool hit = false;
                    V3 a_w, b_w, n;
                    if (vi < nv) {
                        const V3 vw = xpoint(Xm, cmul(ld3(verts + 3 * vi), mscale));
                        const V3 ip = xpoint(Xp_inv, vw);
                        const V3 on_plane = xpoint(Xp, V3(ip.x, ip.y, 0.0f));
                        const float dist = dot(vw - on_plane, pn);
                        if (dist < gap_sum + (marg_m + marg_p)) {
                            // write_contact with its own gap test (collide.py:210-254; radius_eff = 0)
                            const V3 center = (vw + on_plane) * 0.5f;
                            n = unit(-pn);
                            a_w = center - n * (0.5f * dist + 0.0f);
                            b_w = center + n * (0.5f * dist + 0.0f);
                            const float dd = dot(b_w - a_w, n) - (0.0f + 0.0f + marg_m + marg_p);
                            hit = !(dd > gap_sum);
                        }
                    }
                    const unsigned hits = (__ballot_sync(gmask, hit) >> (grp * L)) & (L == 32 ? 0xffffffffu : ((1u << L) - 1u));
                    if (hit) {
                        const int o = slot0 + n_total + written + __popc(hits & ((1u << l) - 1u));
                        const float om_a = 0.0f + marg_m, om_b = 0.0f + marg_p;
                        const V3 p0 = xpoint(Xbw_a, a_w), p1 = xpoint(Xbw_b, b_w);
                        const V3 o0 = xvec(Xbw_a, om_a * n), o1 = xvec(Xbw_b, -om_b * n);
                        cb[CF_BODY_A * T + o] = __int_as_float(body0 >= 0 ? body0 - bs : -1);
                        cb[CF_BODY_B * T + o] = __int_as_float(body1 >= 0 ? body1 - bs : -1);
                        cb[CF_SHAPE0 * T + o] = __int_as_float(msa);
                        cb[CF_SHAPE1 * T + o] = __int_as_float(psb);
                        cb[CF_P0X * T + o] = p0.x; cb[CF_P0Y * T + o] = p0.y; cb[CF_P0Z * T + o] = p0.z;
                        cb[CF_P1X * T + o] = p1.x; cb[CF_P1Y * T + o] = p1.y; cb[CF_P1Z * T + o] = p1.z;
                        cb[CF_O0X * T + o] = o0.x; cb[CF_O0Y * T + o] = o0.y; cb[CF_O0Z * T + o] = o0.z;
                        cb[CF_O1X * T + o] = o1.x; cb[CF_O1Y * T + o] = o1.y; cb[CF_O1Z * T + o] = o1.z;
                        cb[CF_NX * T + o] = n.x; cb[CF_NY * T + o] = n.y; cb[CF_NZ * T + o] = n.z;
                        cb[CF_MARGIN0 * T + o] = om_a;
                        cb[CF_MARGIN1 * T + o] = om_b;
                        cb[CF_MU * T + o] = (d.shape_material_mu[msa] + d.shape_material_mu[psb]) / 2.0f;
                        cb[CF_MU_TORSIONAL * T + o] = (d.shape_material_mu_torsional[msa] + d.shape_material_mu_torsional[psb]) / 2.0f;
                        cb[CF_MU_ROLLING * T + o] = (d.shape_material_mu_rolling[msa] + d.shape_material_mu_rolling[psb]) / 2.0f;
                        cb[CF_KE * T + o] = 0.5f * (d.shape_material_ke[msa] + d.shape_material_ke[psb]);
                        cb[CF_KD * T + o] = 0.5f * (d.shape_material_kd[msa] + d.shape_material_kd[psb]);
                        cb[CF_KF * T + o] = 0.5f * (d.shape_material_kf[msa] + d.shape_material_kf[psb]);
                        cb[CF_KA * T + o] = 0.5f * (d.shape_material_ka[msa] + d.shape_material_ka[psb]);
                    }
                    written += __popc(hits);
                }
                n_total += written;
            }
            seg_lo = seg_hi + 1;
            mesh_lanes &= mesh_lanes - 1;
        }
    }
    if (live && l == 0) M.env_contact_count[env] = n_total;
}

// ---- run-time broad phases: per-world NxN enumeration / sweep-and-prune (reference geometry/broad_phase_nxn.py:132-218,
// broad_phase_sap.py:159-515) ---------------------------------------------------------------------------------------------------
// One sub-warp group per environment, like every kernel of this file.  The reference runs 1 (NxN) or 5 launches + 2 library sorts
// (SAP) over global arrays with a global atomic per candidate; here a world's shapes, their AABBs and - for SAP - their sorted
// projections live in shared memory, and the candidates leave the kernel already in deterministic contact-key order (rank sort by
// (shape_a, shape_b) after the narrow phase's type ordering), which is what lets collide_kernel assign contact slots by prefix sum.
NB2_DEV bool group_pair_collides(int ga, int gb) {  // test_group_pair (broad_phase_common.py:221-238)
    if (ga == 0 || gb == 0) return false;
    if (ga > 0) return ga == gb || gb < 0;
    return ga != gb;
}
struct __align__(8) BpSlot {
    float lo[3], hi[3];
    float disp[3];   // speculative contacts: displacement over the collision-update interval (zero otherwise)
    float pad;
    float plo, phi;  // projection on the SAP axis
    int shape;       // model shape id
    int info;        // bit 0 collides, bit 1 global (world -1), bit 2 immovable (static or kinematic body); group in the high bits is separate
    int group;
    int type;
};
template <int L>
__global__ void __launch_bounds__(32) broadphase_kernel(DevModel M, const float* __restrict__ body_q) {
    constexpr int G = 32 / L;
    extern __shared__ unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, grp = lane / L, l = lane % L;
    const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << (grp * L));
    const int env = blockIdx.x * G + grp;
    const bool live = env < M.env_count;
    const nb2_model_desc& d = M.d;
    const int cap = M.dyn_pair_cap, max_slots = M.max_env_slots_shapes;
    // per group: slots | sort order (SAP) | candidate keys | candidate values | counter
    const size_t per_group = size_t(max_slots) * sizeof(BpSlot) + size_t(max_slots) * sizeof(int) + size_t(cap) * (sizeof(long long) + sizeof(int)) + 16;
    unsigned char* base = smem_raw + size_t(grp) * ((per_group + 15) & ~size_t(15));
    BpSlot* slots = reinterpret_cast<BpSlot*>(base);
    long long* ckey = reinterpret_cast<long long*>(base + ((size_t(max_slots) * sizeof(BpSlot) + 7) & ~size_t(7)));
    int* cval = reinterpret_cast<int*>(ckey + cap);
    int* order = cval + cap;
    int* counter = order + max_slots;
    int ss = 0, nloc = 0, ns = 0;
    if (live) {
        ss = M.env_shape_start[env];
        nloc = M.env_shape_start[env + 1] - ss;
        ns = nloc + M.global_shape_count;
    }
    if (l == 0) *counter = 0;
    const V3 axis = unit(V3(0.5935f, 0.7790f, 0.1235f));  // broad_phase_sap.py:702-703
    for (int s = l; s < ns; s += L) {
        const int sid = s < nloc ? ss + s : M.global_shapes[s - nloc];
        const int body = d.shape_body[sid];
        Xf X = ldx(d.shape_transform + 7 * sid);
        if (body != -1) X = xmul(ldx(body_q + 7 * body), X);
        const int stype = d.shape_type[sid];
        V3 llo, lhi, lo, hi;
        if (stype == GEO_CONVEX_MESH || stype == GEO_MESH) {
            llo = ld3(d.shape_collision_aabb_lower + 3 * sid);
            lhi = ld3(d.shape_collision_aabb_upper + 3 * sid);
        }
        shape_aabb(stype, ld3(d.shape_scale + 3 * sid), X, d.shape_margin[sid] + d.shape_gap[sid], d.shape_collision_radius[sid], llo, lhi, lo, hi);
        BpSlot& r = slots[s];
        V3 disp;
        if (M.spec_mode == 2) disp = shape_motion(M, body_q, sid, body, X, lo, hi).disp;  // also grows the AABB by the angular travel
        st3(r.lo, lo);
        st3(r.hi, hi);
        st3(r.disp, disp);
        // _sap_project_aabb (broad_phase_sap.py:44-80), AABBs pre-expanded (no extra gap)
        const V3 half = 0.5f * (hi - lo);
        const float radius = dot(vabs(axis), half), center = dot(axis, 0.5f * (lo + hi));
        r.plo = center - radius;
        r.phi = center + radius;
        if (M.spec_mode == 2) {  // the interval also covers the displacement along the sort axis, clamped to the extension cap
            const float pd = clamp_w(dot(axis, disp), -M.spec_max_ext, M.spec_max_ext);
            r.plo += fmin_w(pd, 0.0f);
            r.phi += fmax_w(pd, 0.0f);
        }
        r.shape = sid;
        r.group = d.shape_collision_group ? d.shape_collision_group[sid] : 1;
        r.type = stype;
        const bool immovable = body < 0 || (d.body_flags[body] & 2) != 0;
        r.info = ((d.shape_flags[sid] & 2) ? 1 : 0) | (s >= nloc ? 2 : 0) | (immovable ? 4 : 0);
    }
    __syncwarp(gmask);
    // the per-pair filter chain of _nxn_broadphase_kernel / _process_sap_work_package, then the candidate append
    auto consider = [&](int i, int j) {
        const BpSlot& a = slots[i];
        const BpSlot& b = slots[j];
        if (!(a.info & b.info & 1)) return;             // precompute_world_map keeps COLLIDE_SHAPES shapes only
        if ((a.info & 2) && (b.info & 2)) return;       // shared-vs-shared pairs belong to the dedicated segment (no body involved)
        if (!group_pair_collides(a.group, b.group)) return;
        if (!M.include_static_kinematic_pairs && (a.info & 4) && (b.info & 4)) return;
        if (M.spec_mode == 2) {  // check_aabb_overlap_moving: swept over the relative displacement (symmetric in the two shapes)
            if (!aabb_overlap_moving(ld3(a.lo), ld3(a.hi), ld3(b.lo), ld3(b.hi), ld3(a.disp) - ld3(b.disp))) return;
        } else if (!(a.lo[0] <= b.hi[0] && a.hi[0] >= b.lo[0] && a.lo[1] <= b.hi[1] && a.hi[1] >= b.lo[1] && a.lo[2] <= b.hi[2] && a.hi[2] >= b.lo[2]))
            return;
        const int s1 = min(a.shape, b.shape), s2 = max(a.shape, b.shape);
        if (M.filter_count > 0) {  // is_pair_excluded: binary search of the sorted exclusion list
            const long long key = ((long long)s1 << 32) | (long long)s2;
            int lo = 0, hi = M.filter_count - 1;
            while (lo <= hi) {
                const int mid = (lo + hi) >> 1;
                const long long m = M.filter_keys[mid];
                if (m == key) return;
                if (key < m) hi = mid - 1;
                else lo = mid + 1;
            }
        }
        // narrow-phase type ordering (narrow_phase.py:525-528) on the canonical (min, max) pair
        const BpSlot& p1 = a.shape == s1 ? a : b;
        const BpSlot& p2 = a.shape == s1 ? b : a;
        const int i1 = a.shape == s1 ? i : j, i2 = a.shape == s1 ? j : i;
        const bool swap = p1.type > p2.type;
        const int sa = swap ? p2.shape : p1.shape, sb = swap ? p1.shape : p2.shape, ia = swap ? i2 : i1, ib = swap ? i1 : i2;
        const int pos = atomicAdd(counter, 1);
        if (pos < cap) {
            ckey[pos] = ((long long)sa << 32) | (long long)sb;
            cval[pos] = ia | (ib << 16);
        }
    };
    if (M.broad_phase == NB2_BROAD_PHASE_SAP) {
        // sort the world's shapes by projected lower bound (stable rank sort; ties cannot change the candidate set)
        for (int s = l; s < ns; s += L) {
            const float v = slots[s].plo;
            int rank = 0;
            for (int k = 0; k < ns; ++k) rank += (slots[k].plo < v || (slots[k].plo == v && k < s)) ? 1 : 0;
            order[rank] = s;
        }
        __syncwarp(gmask);
        for (int i = l; i < ns; i += L) {  // _sap_range_kernel: sweep while lower_j < upper_i
            const int si = order[i];
            const float upper = slots[si].phi;
            for (int j = i + 1; j < ns; ++j) {
                const int sj = order[j];
                if (!(slots[sj].plo < upper)) break;
                consider(si, sj);
            }
        }
    } else {
        for (int i = 0; i < ns; ++i)  // _nxn_broadphase_kernel: every pair of the world's slice
            for (int j = i + 1 + l; j < ns; j += L) consider(i, j);
    }
    __syncwarp(gmask);
    const int total = *counter, n = min(total, cap);
    // rank sort by the deterministic contact key (keys are unique: one entry per shape pair)
    if (live) {
        int2* out = M.dyn_pairs + size_t(env) * cap;
        for (int c = l; c < n; c += L) {
            const long long key = ckey[c];
            int rank = 0;
            for (int k = 0; k < n; ++k) rank += ckey[k] < key ? 1 : 0;
            out[rank] = make_int2(cval[c] & 0xffff, cval[c] >> 16);
        }
        if (l == 0) M.env_dyn_count[env] = total;
    }
}

// ---- export to the reference `Contacts` arrays ---------------------------------------------------
// Single-CTA exclusive scan of the per-env counts (E <= a few 10^5), then one group per env scatters its block.
__global__ void __launch_bounds__(1024) contact_scan_kernel(const int* __restrict__ counts, int E, int* __restrict__ offsets,
                                                            int* __restrict__ rigid_contact_count) {
    __shared__ int warp_sums[32];
    __shared__ int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int base = 0; base < E; base += 1024) {
        int i = base + threadIdx.x;
        int v = i < E ? counts[i] : 0;
        int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warp_sums[threadIdx.x >> 5] = incl;
        __syncthreads();
        if (threadIdx.x < 32) {
            int w = warp_sums[threadIdx.x];
            int wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                int t = __shfl_up_sync(0xffffffffu, wi, o);
                if (threadIdx.x >= o) wi += t;
            }
            warp_sums[threadIdx.x] = wi - w;
        }
        __syncthreads();
        int excl = carry + warp_sums[threadIdx.x >> 5] + incl - v;
        if (i < E) offsets[i] = excl;
        __syncthreads();
        if (threadIdx.x == 1023) carry = excl + v;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        offsets[E] = carry;
        if (rigid_contact_count) rigid_contact_count[0] = carry;
    }
}

// SELF_SCAN (batches up to 8192 environments): one pass - every CTA (4 environments, one warp each) first sums the contact
// counts of all environments before its own (E/128 coalesced int loads per thread out of L2; exact integer arithmetic, so
// the offsets equal the scan's) and then scatters its environments' contact blocks; this saves the single-CTA scan launch
// (6 us of a 40 us collide stage at 4096 envs).  The sum is O(E^2 / 128) over the grid, so larger batches keep the
// separate contact_scan_kernel and read its offsets.
template <bool SELF_SCAN>
__global__ void __launch_bounds__(128) contact_export_kernel(DevModel M, nb2_contacts_view out) {
    __shared__ int warp_part[4];
    const int env0 = blockIdx.x * 4;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int env = env0 + wid;
    int dst0;
    if (SELF_SCAN) {
        int part = 0;
        for (int i = threadIdx.x; i < env0; i += 128) part += M.env_contact_count[i];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
        if (lane == 0) warp_part[wid] = part;
        __syncthreads();
        dst0 = warp_part[0] + warp_part[1] + warp_part[2] + warp_part[3];
        for (int e = env0; e < env && e < M.env_count; ++e) dst0 += M.env_contact_count[e];
    } else {
        dst0 = env < M.env_count ? M.env_contact_offset[env] : 0;
    }
    if (env >= M.env_count) return;
    const int n = M.env_contact_count[env];
    if (SELF_SCAN && lane == 0) {
        M.env_contact_offset[env] = dst0;
        if (env == M.env_count - 1) {
            M.env_contact_offset[M.env_count] = dst0 + n;
            out.rigid_contact_count[0] = dst0 + n;
        }
    }
    const int src0 = M.env_slot_start[env];
    const size_t T = size_t(M.slot_total);
    const float* cb = M.cb;
    for (int c = lane; c < n; c += 32) {
        const int s = src0 + c, o = dst0 + c;
        if (o >= out.rigid_contact_max) break;  // overflow: count keeps growing, writes dropped (collide.py:176-177)
        out.shape0[o] = __float_as_int(cb[CF_SHAPE0 * T + s]);
        out.shape1[o] = __float_as_int(cb[CF_SHAPE1 * T + s]);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            out.point0[3 * o + k] = cb[(CF_P0X + k) * T + s];
            out.point1[3 * o + k] = cb[(CF_P1X + k) * T + s];
            out.offset0[3 * o + k] = cb[(CF_O0X + k) * T + s];
            out.offset1[3 * o + k] = cb[(CF_O1X + k) * T + s];
            out.normal[3 * o + k] = cb[(CF_NX + k) * T + s];
        }
        out.margin0[o] = cb[CF_MARGIN0 * T + s];
        out.margin1[o] = cb[CF_MARGIN1 * T + s];
        if (out.tids) out.tids[o] = 0;
    }
}

// ---- deterministic=True: reorder the exported arrays into the reference's global sort-key order (nb2_contacts_sort) -----------
__global__ void __launch_bounds__(256) sort_keys_kernel(nb2_contacts_view c, unsigned long long shape_radix, unsigned long long* __restrict__ keys,
                                                        int* __restrict__ idx, float* __restrict__ stage) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= c.rigid_contact_max) return;
    const int n = min(c.rigid_contact_count[0], c.rigid_contact_max);
    idx[i] = i;
    if (i >= n) {
        keys[i] = ~0ull;
        return;
    }
    // make_contact_sort_key orders by (shape_a, shape_b, sub_key); the export already lists a pair's contacts in sub-key order
    keys[i] = (unsigned long long)(unsigned)c.shape0[i] * shape_radix + (unsigned long long)(unsigned)c.shape1[i];
    float* st = stage + size_t(i) * 20;
    st[0] = __int_as_float(c.shape0[i]);
    st[1] = __int_as_float(c.shape1[i]);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        st[2 + k] = c.point0[3 * i + k];
        st[5 + k] = c.point1[3 * i + k];
        st[8 + k] = c.offset0[3 * i + k];
        st[11 + k] = c.offset1[3 * i + k];
        st[14 + k] = c.normal[3 * i + k];
    }
    st[17] = c.margin0[i];
    st[18] = c.margin1[i];
    st[19] = c.tids ? __int_as_float(c.tids[i]) : 0.0f;
}

__global__ void __launch_bounds__(256) sort_gather_kernel(nb2_contacts_view c, const int* __restrict__ idx_sorted, const float* __restrict__ stage,
                                                          int* __restrict__ rank) {
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= c.rigid_contact_max) return;
    const int n = min(c.rigid_contact_count[0], c.rigid_contact_max);
    if (p >= n) return;
    const int i = idx_sorted[p];  // exported index that lands at position p
    rank[i] = p;
    const float* st = stage + size_t(i) * 20;
    c.shape0[p] = __float_as_int(st[0]);
    c.shape1[p] = __float_as_int(st[1]);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        c.point0[3 * p + k] = st[2 + k];
        c.point1[3 * p + k] = st[5 + k];
        c.offset0[3 * p + k] = st[8 + k];
        c.offset1[3 * p + k] = st[11 + k];
        c.normal[3 * p + k] = st[14 + k];
    }
    c.margin0[p] = st[17];
    c.margin1[p] = st[18];
    if (c.tids) c.tids[p] = __float_as_int(st[19]);
}

nb2_status launch_contacts_sort(nb2_model* m, const nb2_contacts_view& c, cudaStream_t s) {
    const int C = c.rigid_contact_max;
    if (C == 0) return NB2_OK;
    int bits = 1;
    while ((1ull << bits) <= (unsigned long long)m->dev.d.shape_count) ++bits;  // shape ids are 0 .. shape_count - 1
    const unsigned long long radix = 1ull << bits;
    const int end_bit = 2 * bits < 64 ? 2 * bits : 64;
    if (C > m->sort_capacity) {
        size_t temp = 0;
        NB2_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, temp, (const unsigned long long*)nullptr, (unsigned long long*)nullptr,
                                                       (const int*)nullptr, (int*)nullptr, C, 0, end_bit, s));
        void *k = nullptr, *ix = nullptr, *st = nullptr, *tmp = nullptr, *rk = nullptr;
        NB2_CUDA_CHECK(cudaMalloc(&k, size_t(C) * 2 * sizeof(unsigned long long)));
        NB2_CUDA_CHECK(cudaMalloc(&ix, size_t(C) * 2 * sizeof(int)));
        NB2_CUDA_CHECK(cudaMalloc(&st, size_t(C) * 20 * sizeof(float)));
        NB2_CUDA_CHECK(cudaMalloc(&rk, size_t(C) * sizeof(int)));
        NB2_CUDA_CHECK(cudaMalloc(&tmp, std::max<size_t>(temp, 16)));
        for (void* p : {k, ix, st, rk, tmp}) m->allocations.push_back(p);
        m->sort_keys = static_cast<unsigned long long*>(k);
        m->sort_keys_sorted = m->sort_keys + C;
        m->sort_idx = static_cast<int*>(ix);
        m->sort_idx_sorted = m->sort_idx + C;
        m->sort_stage = static_cast<float*>(st);
        m->sort_rank = static_cast<int*>(rk);
        m->sort_temp = tmp;
        m->sort_temp_bytes = temp;
        m->sort_capacity = C;
    }
    sort_keys_kernel<<<(C + 255) / 256, 256, 0, s>>>(c, radix, m->sort_keys, m->sort_idx, m->sort_stage);
    size_t temp = m->sort_temp_bytes;
    NB2_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(m->sort_temp, temp, m->sort_keys, m->sort_keys_sorted, m->sort_idx, m->sort_idx_sorted, C, 0,
                                                   end_bit, s));  // stable
    sort_gather_kernel<<<(C + 255) / 256, 256, 0, s>>>(c, m->sort_idx_sorted, m->sort_stage, m->sort_rank);
    m->dev.export_rank = m->sort_rank;
    count_launch(2);
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

// ---- import of a foreign reference-layout Contacts buffer into the contact blocks (nb2_contacts_import) ----------------------
__global__ void __launch_bounds__(256) import_keys_kernel(DevModel M, nb2_contacts_view in, int implicit_single, int* __restrict__ keys,
                                                          int* __restrict__ idx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= in.rigid_contact_max) return;
    const nb2_model_desc& d = M.d;
    const int n = min(in.rigid_contact_count[0], in.rigid_contact_max);
    int key = M.env_count;  // sentinel: sorts behind every environment
    if (i < n) {
        const int s0 = in.shape0[i], s1 = in.shape1[i];
        if (s0 >= 0 && s1 >= 0 && s0 != s1 && s0 < d.shape_count && s1 < d.shape_count) {
            const bool dynamic = d.shape_body[s0] >= 0 || d.shape_body[s1] >= 0;  // static-vs-static contacts move nothing
            int env = 0;
            if (!implicit_single) {
                const int w0 = d.shape_world[s0], w1 = d.shape_world[s1];
                env = w0 >= 0 ? w0 : w1;
            }
            if (dynamic && env >= 0 && env < M.env_count) key = env;
        }
    }
    keys[i] = key;
    idx[i] = i;
}

NB2_DEV int lower_bound_int(const int* a, int n, int v) {
    int lo = 0, hi = n;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (a[mid] < v) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(128) import_scatter_kernel(DevModel M, nb2_contacts_view in, const int* __restrict__ keys_sorted,
                                                             const int* __restrict__ idx_sorted) {
    const int env = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (env >= M.env_count) return;
    const int lane = threadIdx.x & 31;
    const nb2_model_desc& d = M.d;
    const int first = lower_bound_int(keys_sorted, in.rigid_contact_max, env);
    const int last = lower_bound_int(keys_sorted, in.rigid_contact_max, env + 1);
    const int slot0 = M.env_slot_start[env], cap = M.env_slot_start[env + 1] - slot0;
    const int n = min(last - first, cap);  // beyond the block capacity: dropped, like every other overflow of this path
    if (lane == 0) M.env_contact_count[env] = n;
    const int bs = M.env_body_start[env];
    float* cb = M.cb;
    const size_t T = size_t(M.slot_total);
    for (int c = lane; c < n; c += 32) {
        const int i = idx_sorted[first + c], slot = slot0 + c;
        const int sa = in.shape0[i], sb = in.shape1[i];
        const int body0 = d.shape_body[sa], body1 = d.shape_body[sb];
        cb[CF_BODY_A * T + slot] = __int_as_float(body0 >= 0 ? body0 - bs : -1);
        cb[CF_BODY_B * T + slot] = __int_as_float(body1 >= 0 ? body1 - bs : -1);
        cb[CF_SHAPE0 * T + slot] = __int_as_float(sa);
        cb[CF_SHAPE1 * T + slot] = __int_as_float(sb);
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            cb[(CF_P0X + k) * T + slot] = in.point0[3 * i + k];
            cb[(CF_P1X + k) * T + slot] = in.point1[3 * i + k];
            cb[(CF_O0X + k) * T + slot] = in.offset0[3 * i + k];
            cb[(CF_O1X + k) * T + slot] = in.offset1[3 * i + k];
            cb[(CF_NX + k) * T + slot] = in.normal[3 * i + k];
        }
        cb[CF_MARGIN0 * T + slot] = in.margin0[i];
        cb[CF_MARGIN1 * T + slot] = in.margin1[i];
        // pair-averaged coefficients, exactly as the collide kernel's write-out computes them
        cb[CF_MU * T + slot] = (d.shape_material_mu[sa] + d.shape_material_mu[sb]) / 2.0f;
        cb[CF_MU_TORSIONAL * T + slot] = (d.shape_material_mu_torsional[sa] + d.shape_material_mu_torsional[sb]) / 2.0f;
        cb[CF_MU_ROLLING * T + slot] = (d.shape_material_mu_rolling[sa] + d.shape_material_mu_rolling[sb]) / 2.0f;
        cb[CF_KE * T + slot] = 0.5f * (d.shape_material_ke[sa] + d.shape_material_ke[sb]);
        cb[CF_KD * T + slot] = 0.5f * (d.shape_material_kd[sa] + d.shape_material_kd[sb]);
        cb[CF_KF * T + slot] = 0.5f * (d.shape_material_kf[sa] + d.shape_material_kf[sb]);
        cb[CF_KA * T + slot] = 0.5f * (d.shape_material_ka[sa] + d.shape_material_ka[sb]);
    }
}

nb2_status launch_contacts_import(nb2_model* m, const nb2_contacts_view& in, cudaStream_t s) {
    const DevModel& M = m->dev;
    if (M.env_count == 0) return NB2_OK;
    const int C = in.rigid_contact_max;
    int end_bit = 1;
    while ((1 << end_bit) <= M.env_count) ++end_bit;  // keys are 0..env_count
    if (C > m->import_capacity) {  // (re)allocate scratch: not capturable, see the header
        size_t temp = 0;
        NB2_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(nullptr, temp, (const int*)nullptr, (int*)nullptr, (const int*)nullptr, (int*)nullptr, C, 0,
                                                       end_bit, s));
        int* buf = nullptr;
        NB2_CUDA_CHECK(cudaMalloc(&buf, size_t(C) * 4 * sizeof(int)));
        m->allocations.push_back(buf);
        void* tmp = nullptr;
        NB2_CUDA_CHECK(cudaMalloc(&tmp, std::max<size_t>(temp, 16)));
        m->allocations.push_back(tmp);
        m->import_keys = buf;
        m->import_keys_sorted = buf + C;
        m->import_idx = buf + 2 * size_t(C);
        m->import_idx_sorted = buf + 3 * size_t(C);
        m->import_temp = tmp;
        m->import_temp_bytes = temp;
        m->import_capacity = C;
    }
    if (C > 0) {
        import_keys_kernel<<<(C + 255) / 256, 256, 0, s>>>(M, in, m->implicit_single ? 1 : 0, m->import_keys, m->import_idx);
        size_t temp = m->import_temp_bytes;
        NB2_CUDA_CHECK(cub::DeviceRadixSort::SortPairs(m->import_temp, temp, m->import_keys, m->import_keys_sorted, m->import_idx,
                                                       m->import_idx_sorted, C, 0, end_bit, s));  // stable: array order kept per env
    }
    import_scatter_kernel<<<(M.env_count + 3) / 4, 128, 0, s>>>(M, in, m->import_keys_sorted, m->import_idx_sorted);
    count_launch(2);
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

template <int L, bool CONVEX, int WARPS>
static nb2_status launch_collide_W(nb2_model* m, const float* body_q, cudaStream_t s) {
    const DevModel& M = m->dev;
    const int NE = (32 / L) * WARPS;
    const int blocks = (M.env_count + NE - 1) / NE;
    const size_t smem = size_t(NE) * (M.max_env_slots_shapes * (sizeof(SlotRec) + (CONVEX && M.spec_mode != 0 ? sizeof(SlotMotionRec) : 0)) +
                                      stage_bytes_per_group(L));
    if (smem > 48 * 1024)
        NB2_CUDA_CHECK(cudaFuncSetAttribute(collide_kernel<L, CONVEX, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    collide_kernel<L, CONVEX, WARPS><<<blocks, 32 * WARPS, smem, s>>>(M, body_q);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

// warps per CTA: 8 when the batch puts at least 8 warps on every SM, shared memory permitting
template <int L, bool CONVEX>
static nb2_status launch_collide_L(nb2_model* m, const float* body_q, cudaStream_t s) {
    const DevModel& M = m->dev;
    const size_t per_warp = size_t(32 / L) * (M.max_env_slots_shapes * (sizeof(SlotRec) + (CONVEX && M.spec_mode != 0 ? sizeof(SlotMotionRec) : 0)) +
                                              stage_bytes_per_group(L));
    if (per_warp > 200 * 1024) {
        set_error("collide: too many shapes per environment for the fused kernel");
        return NB2_ERR_CAPACITY;
    }
    if (warps_per_sm(m, L) >= 8 && per_warp * 8 <= 200 * 1024) return launch_collide_W<L, CONVEX, 8>(m, body_q, s);
    return launch_collide_W<L, CONVEX, 1>(m, body_q, s);
}

template <int L>
static nb2_status launch_broadphase_L(nb2_model* m, const float* body_q, cudaStream_t s) {
    const DevModel& M = m->dev;
    const int G = 32 / L;
    const size_t per_group = size_t(M.max_env_slots_shapes) * sizeof(BpSlot) + size_t(M.max_env_slots_shapes) * sizeof(int) +
                             size_t(M.dyn_pair_cap) * (sizeof(long long) + sizeof(int)) + 16;
    const size_t smem = ((per_group + 15) & ~size_t(15)) * G;
    if (smem > 200 * 1024) {
        set_error("broad phase: too many shapes / candidate pairs per world for the shared-memory sweep (lower max_pairs_per_world)");
        return NB2_ERR_CAPACITY;
    }
    if (smem > 48 * 1024) NB2_CUDA_CHECK(cudaFuncSetAttribute(broadphase_kernel<L>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    broadphase_kernel<L><<<(M.env_count + G - 1) / G, 32, smem, s>>>(M, body_q);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

nb2_status launch_broadphase(nb2_model* m, const float* body_q, cudaStream_t s) {
    if (m->dev.env_count == 0 || m->dev.d.shape_count == 0) return NB2_OK;
    switch (m->lanes_per_env) {
        case 8: return launch_broadphase_L<8>(m, body_q, s);
        case 16: return launch_broadphase_L<16>(m, body_q, s);
        default: return launch_broadphase_L<32>(m, body_q, s);
    }
}

nb2_status launch_collide(nb2_model* m, const float* body_q, const nb2_contacts_view* contacts, cudaStream_t s) {
    const DevModel& M = m->dev;
    if (M.env_count == 0 || M.d.shape_count == 0) return NB2_OK;
    nb2_status st;
    if (contacts && (!contacts->rigid_contact_count || !contacts->shape0 || !contacts->shape1 || !contacts->point0 || !contacts->point1 ||
                     !contacts->offset0 || !contacts->offset1 || !contacts->normal || !contacts->margin0 || !contacts->margin1)) {
        set_error("nb2_collide: contacts view has NULL arrays");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (m->has_mesh_pairs && M.spec_mode != 0) {
        set_error("nb2_collide_speculative: MESH shapes are not supported with speculative contacts");
        return NB2_ERR_UNSUPPORTED;
    }
    if (M.dyn_pairs && (st = launch_broadphase(m, body_q, s)) != NB2_OK) return st;
    // speculative contacts and mesh-plane pairs live in the generic (CONVEX = true) instantiation only
    const bool generic = m->has_convex_pairs || M.spec_mode != 0 || m->has_mesh_pairs;
#define COLLIDE_DISPATCH(LANES) st = generic ? launch_collide_L<LANES, true>(m, body_q, s) : launch_collide_L<LANES, false>(m, body_q, s)
    switch (m->lanes_per_env) {
        case 8: COLLIDE_DISPATCH(8); break;
        case 16: COLLIDE_DISPATCH(16); break;
        default: COLLIDE_DISPATCH(32); break;
    }
#undef COLLIDE_DISPATCH
    if (st != NB2_OK) return st;
    // The `Contacts` arrays are written by a second kernel.  Writing them from collide_kernel itself, with a decoupled look-back for
    // the offsets, lost: 690.1 vs 678.3 us per 4096-quadruped frame (profiles/r2j_fused_export_ab.txt, DESIGN.md section 2).
    if (contacts) {
        if (M.env_count <= 8192) {
            contact_export_kernel<true><<<(M.env_count + 3) / 4, 128, 0, s>>>(M, *contacts);
            count_launch();
        } else {
            contact_scan_kernel<<<1, 1024, 0, s>>>(M.env_contact_count, M.env_count, M.env_contact_offset, contacts->rigid_contact_count);
            contact_export_kernel<false><<<(M.env_count + 3) / 4, 128, 0, s>>>(M, *contacts);
            count_launch(2);
        }
        NB2_CUDA_CHECK(cudaGetLastError());
    }
    return NB2_OK;
}

}  // namespace nb2
