// nb2_xpbd.cu - fused XPBD rigid-body substep for sm_100a (reference SolverXPBD.step, solver_xpbd.py:329-862).
//
// The reference runs `2 + iterations*6 + 1` kernel launches per substep, each re-reading body state from
// HBM/L2 and summing per-body corrections with float atomics.  Here ONE launch does the whole substep for
// every environment: a sub-warp group of L lanes owns one environment (a CTA is one warp = 32/L environments),
// body state lives in shared memory for the entire Jacobi loop, and the atomics are replaced by ordered
// per-body sums (contacts in contact order, joints in joint order, parent before child) - which is exactly the
// order the reference's serial CPU device produces, so results are run-to-run deterministic.
//
//   apply_joint_forces            kernels.py:945-1075     joint lanes -> ordered per-body sum into body_f copy
//   integrate_bodies              solver.py:112-170       body lanes
//   per iteration:
//     solve_body_contact_positions  kernels.py:2164-2399  contact lanes -> smem delta records
//     apply_body_deltas (weighted)  kernels.py:864-933    body lanes, ordered sum over the env's contacts
//     solve_body_joints             kernels.py:1513-2044  joint lanes -> smem delta records
//     apply_body_deltas             kernels.py:864-933    body lanes, ordered sum over the body's joints (CSR)
//   copy_kinematic_body_state      kernels.py:19-32       implicit: kinematic bodies are never modified
#include "nb2_internal.cuh"
#include "nb2_math.cuh"

#define NB2_GPU __device__ __forceinline__

namespace nb2 {

enum { JT_PRISMATIC = 0, JT_REVOLUTE = 1, JT_BALL = 2, JT_FIXED = 3, JT_FREE = 4, JT_DISTANCE = 5, JT_D6 = 6, JT_ROD = 7 };
enum { BODY_KINEMATIC = 2 };

// shared-memory body record (floats): odd stride -> consecutive bodies hit different banks
enum { BR_Q = 0, BR_QD = 7, BR_COM = 13, BR_INVM = 16, BR_INVI = 17, BR_I = 26, BR_SIZE = 35 };
enum { DR_SIZE = 13 };  // delta record: lin_a, ang_a, lin_b, ang_b, active
// per-contact constants of the Jacobi loop, staged once per substep: point0, point1, normal, margin0 + margin1, the three friction
// coefficients and the friction anchors point + offset (odd stride: lanes = consecutive contacts)
enum { CC_P0 = 0, CC_P1 = 3, CC_N = 6, CC_MSUM = 9, CC_MU = 10, CC_MUT = 11, CC_MUR = 12, CC_Q0 = 13, CC_Q1 = 16, CC_SIZE = 19 };

// Code size.  With 14-warp CTAs walking the code together the instruction stream is fetched once per CTA, so the helpers are inlined
// and the 3-row joint loops unrolled: no per-row component selects / loop control, three independent rows for the scheduler to
// interleave.  Unrolled rows: 143.7 -> 139.7 us at 4096 quadruped envs (profiles/r2j_fused_export_ab.txt).

struct BodyView {
    Xf X;
    V3 com;
    float inv_m;
    const float* rec;  // shared-memory record (inverse inertia is read from it on demand); nullptr = the static world
    V3 v, w;
};

NB2_DEV BodyView load_body(const float* rec) {
    BodyView b;
    b.X = ldx(rec + BR_Q);
    b.v = ld3(rec + BR_QD);
    b.w = ld3(rec + BR_QD + 3);
    b.com = ld3(rec + BR_COM);
    b.inv_m = rec[BR_INVM];
    b.rec = rec;
    return b;
}
NB2_DEV BodyView static_body() {  // body index -1: the world
    BodyView b;
    b.inv_m = 0.f;
    b.rec = nullptr;
    return b;
}

// r^T I^-1 r with r = ang rotated into the body frame: the angular term of the generalized inverse mass.  For the static
// world the reference multiplies by a zero inverse inertia; the sum is +-0 and adding it leaves the denominator unchanged.
NB2_DEV float ang_inv_mass(const float* rec, V3 ang) {
    if (rec == nullptr) return 0.0f;
    const Q4 q(rec[BR_Q + 3], rec[BR_Q + 4], rec[BR_Q + 5], rec[BR_Q + 6]);
    const V3 r = qrot_inv(q, ang);
    return dot(r, mv(ldm(rec + BR_INVI), r));
}

// shared denominators of compute_contact_constraint_delta / compute_positional_correction (kernels.py:2063-2075)
NB2_DEV float generalized_inv_mass(const BodyView& a, const BodyView& b, V3 lin_a, V3 lin_b, V3 ang_a, V3 ang_b) {
    float denom = 0.0f;
    denom += len2(lin_a) * a.inv_m;
    denom += len2(lin_b) * b.inv_m;
    denom += ang_inv_mass(a.rec, ang_a);
    denom += ang_inv_mass(b.rec, ang_b);
    return denom;
}
NB2_DEV float contact_delta(float err, const BodyView& a, const BodyView& b, V3 lin_a, V3 lin_b, V3 ang_a, V3 ang_b, float relaxation,
                            float dt) {
    float denom = generalized_inv_mass(a, b, lin_a, lin_b, ang_a, ang_b);
    float dl = -err;
    if (denom > 0.0f) dl /= dt * denom;
    return dl * relaxation;
}
// `alpha_dt` is compliance / dt, passed in so that the quotient of the kernel-wide compliance is formed once per substep
NB2_DEV float positional_correction(float err, float derr, const BodyView& a, const BodyView& b, V3 lin_a, V3 lin_b, V3 ang_a, V3 ang_b,
                                    float compliance, float damping, float dt, float alpha_dt) {
    float denom = generalized_inv_mass(a, b, lin_a, lin_b, ang_a, ang_b);
    float alpha = compliance, gamma = compliance * damping;
    float dl = -(err + alpha * 0.0f + gamma * derr);
    if (denom + alpha > 0.0f) dl /= (dt + gamma) * denom + alpha_dt;
    return dl;
}
NB2_DEV float angular_correction(float err, float derr, const BodyView& a, const BodyView& b, V3 ang_a, V3 ang_b, float compliance,
                                 float damping, float dt, float alpha_dt) {
    float denom = 0.0f;
    denom += ang_inv_mass(a.rec, ang_a);
    denom += ang_inv_mass(b.rec, ang_b);
    float alpha = compliance, gamma = compliance * damping;
    float dl = -(err + alpha * 0.0f + gamma * derr);
    if (denom + alpha > 0.0f) dl /= (dt + gamma) * denom + alpha_dt;
    return dl;
}

struct AxisSetup {
    V3 lim_lo, lim_up, target_pos, stiffness, target_vel, damping;
};
// "compute joint target, stiffness, damping" (kernels.py:1691-1751 linear, :1911-1973 angular)
NB2_DEV AxisSetup gather_axes(const nb2_model_desc& d, const nb2_control_view& ctl, int axis_start, int target_start, int offset,
                              int count) {
    AxisSetup s;
    V3 pos_t, pos_w, vel_t, vel_w;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        if (count > k) {
            int ai = axis_start + offset + k, ti = target_start + offset + k;
            V3 axis = ld3(d.joint_axis + 3 * ai);
            V3 lo_t = axis * d.joint_limit_lower[ai], up_t = axis * d.joint_limit_upper[ai];
            V3 lo = vmin(lo_t, up_t), up = vmax(lo_t, up_t);
            if (k == 0) {
                s.lim_lo = lo;
                s.lim_up = up;
            } else {
                s.lim_lo = vmin(s.lim_lo, lo);
                s.lim_up = vmax(s.lim_up, up);
            }
            float ke = d.joint_target_ke[ai], kd = d.joint_target_kd[ai];
            if (ke > 0.0f) {
                V3 wa = axis * ke;
                pos_t += wa * ctl.joint_target_q[ti];
                pos_w += vabs(wa);
            }
            if (kd > 0.0f) {
                V3 wa = axis * kd;
                vel_t += wa * ctl.joint_target_qd[ai];
                vel_w += vabs(wa);
            }
        }
    }
    s.target_pos = pos_t;
    s.stiffness = pos_w;
    s.target_vel = vel_t;
    s.damping = vel_w;
    if (s.stiffness.x > 0.0f) s.target_pos.x /= s.stiffness.x;
    if (s.stiffness.y > 0.0f) s.target_pos.y /= s.stiffness.y;
    if (s.stiffness.z > 0.0f) s.target_pos.z /= s.stiffness.z;
    if (s.damping.x > 0.0f) s.target_vel.x /= s.damping.x;
    if (s.damping.y > 0.0f) s.target_vel.y /= s.damping.y;
    if (s.damping.z > 0.0f) s.target_vel.z /= s.damping.z;
    return s;
}

struct Deltas {
    V3 lin_p, ang_p, lin_c, ang_c;
};

// solve_body_joints for one joint (kernels.py:1513-2044).  `bodies` = this env's shared-memory records.
// Per-joint quantities that do not change over the Jacobi iterations, staged once per substep in shared memory when it
// fits next to the body records without costing a resident CTA: the two joint frames and the angular AxisSetup.
// ... and the joint's integer header (type, enabled, dof counts, child / parent, axis and target offsets), so the
// iteration loop issues no global loads for joint data at all.
enum { JC_XP = 0, JC_XC = 7, JC_ANG = 14, JC_HDR = 32, JC_CHILD = 33, JC_PARENT = 34, JC_AXIS = 35, JC_TARGET = 36,
       JC_SIZE = 37 };  // odd stride: consecutive joints (lanes) hit different banks
NB2_DEV int jc_int(const float* jc, int k) { return reinterpret_cast<const int*>(jc)[k]; }
NB2_DEV void store_axis_setup(float* p, const AxisSetup& s) {
    st3(p, s.lim_lo); st3(p + 3, s.lim_up); st3(p + 6, s.target_pos); st3(p + 9, s.stiffness); st3(p + 12, s.target_vel); st3(p + 15, s.damping);
}
NB2_DEV AxisSetup load_axis_setup(const float* p) {
    AxisSetup s;
    s.lim_lo = ld3(p); s.lim_up = ld3(p + 3); s.target_pos = ld3(p + 6); s.stiffness = ld3(p + 9); s.target_vel = ld3(p + 12); s.damping = ld3(p + 15);
    return s;
}

NB2_DEV bool solve_joint(const nb2_model_desc& d, const nb2_control_view& ctl, const nb2_xpbd_params& P, int j, int body0,
                         const float* bodies, const float* jc, float dt, float lin_alpha_dt, float ang_alpha_dt, Deltas& out) {
    // header: bits 0-3 type, bit 4 enabled, bits 8-11 / 12-15 linear / angular dof counts
    const int hdr = jc ? jc_int(jc, JC_HDR)
                       : (d.joint_type[j] | (d.joint_enabled[j] ? 16 : 0) | (d.joint_dof_dim[2 * j] << 8) | (d.joint_dof_dim[2 * j + 1] << 12));
    const int type = hdr & 15;
    if (!(hdr & 16) || type == JT_FREE) return false;
    const int id_c = (jc ? jc_int(jc, JC_CHILD) : d.joint_child[j]) - body0;
    const int id_p_raw = jc ? jc_int(jc, JC_PARENT) : d.joint_parent[j];
    const int id_p = id_p_raw >= 0 ? id_p_raw - body0 : -1;
    const Xf X_pj = jc ? ldx(jc + JC_XP) : ldx(d.joint_X_p + 7 * j), X_cj = jc ? ldx(jc + JC_XC) : ldx(d.joint_X_c + 7 * j);
    BodyView bp = static_body();
    Xf X_wp = X_pj;
    Xf pose_p = X_pj;
    if (id_p >= 0) {
        bp = load_body(bodies + id_p * BR_SIZE);
        pose_p = bp.X;
        X_wp = xmul(pose_p, X_wp);
    } else {
        bp.X = pose_p;  // tf_a of the correction helpers is pose_p = X_pj for world-attached joints
    }
    BodyView bc = load_body(bodies + id_c * BR_SIZE);
    const Xf pose_c = bc.X;
    const Xf X_wc = xmul(pose_c, X_cj);
    if (bp.inv_m == 0.0f && bc.inv_m == 0.0f) return false;
    V3 lin_dp, ang_dp, lin_dc, ang_dc;
    const Xf rel_pose = xmul(xinv(X_wp), X_wc);
    const V3 rel_p = rel_pose.p;
    const V3 x_p = X_wp.p, x_c = X_wc.p;
    const int axis_start = jc ? jc_int(jc, JC_AXIS) : d.joint_qd_start[j];
    const int target_start = jc ? jc_int(jc, JC_TARGET) : d.joint_target_q_start[j];
    const int lin_count = (hdr >> 8) & 15, ang_count = (hdr >> 12) & 15;
    const V3 wcom_p = xpoint(pose_p, bp.com);
    const V3 wcom_c = xpoint(pose_c, bc.com);
    const V3 vel_p = bp.v, omega_p = bp.w, vel_c = bc.v, omega_c = bc.w;

    if (type == JT_DISTANCE) {
        V3 r_p = x_p - wcom_p, r_c = x_c - wcom_c;
        float lower = d.joint_limit_lower[axis_start], upper = d.joint_limit_upper[axis_start];
        if (lower < 0.0f && upper < 0.0f) return false;
        V3 ad = x_c - x_p;
        float dist = len(ad);
        float err = 0.0f;
        if (lower >= 0.0f && dist < lower) err = dist - lower;
        else if (upper >= 0.0f && dist > upper) err = dist - upper;
        if (fabsf(err) > 1e-9f) {
            V3 lc;
            if (dist > 1e-9f) lc = ad / dist;
            else {
                V3 cd = wcom_c - wcom_p;
                lc = len2(cd) > 1e-18f ? unit(cd) : xvec(X_wp, V3(1.f, 0.f, 0.f));
            }
            V3 lp = -lc, ap = -cross(r_p, lc), ac = cross(r_c, lc);
            float derr = dot(lp, vel_p) + dot(lc, vel_c) + dot(ap, omega_p) + dot(ac, omega_c);
            float compliance = P.joint_linear_compliance, alpha_dt = lin_alpha_dt;
            float ke = d.joint_target_ke[axis_start];
            if (ke > 0.0f) {
                compliance = 1.0f / ke;
                alpha_dt = compliance / dt;
            }
            float damping = d.joint_target_kd[axis_start];
            float dl = positional_correction(err, derr, bp, bc, lp, lc, ap, ac, compliance, damping, dt, alpha_dt);
            lin_dp += lp * (dl * P.joint_linear_relaxation);
            ang_dp += ap * (dl * P.joint_angular_relaxation);
            lin_dc += lc * (dl * P.joint_linear_relaxation);
            ang_dc += ac * (dl * P.joint_angular_relaxation);
        }
    } else {
        const AxisSetup s = gather_axes(d, ctl, axis_start, target_start, 0, lin_count);
        V3 proj = rel_p;
#pragma unroll
        for (int dim = 0; dim < 3; ++dim) {
            float lo = s.lim_lo.get(dim), up = s.lim_up.get(dim), e = rel_p.get(dim);
            if (e < lo) proj.set(dim, lo);
            else if (e > up) proj.set(dim, up);
            else if (s.stiffness.get(dim) > 0.0f) proj.set(dim, clamp_w(s.target_pos.get(dim), lo, up));
        }
        const V3 r_p = xpoint(X_wp, proj) - wcom_p;
        const V3 r_c = x_c - wcom_c;
#pragma unroll
        for (int dim = 0; dim < 3; ++dim) {
            float e = rel_p.get(dim);
            // column `dim` of quat_to_matrix(X_wp.q), i.e. the rotated basis vector
            V3 lc = qrot(X_wp.q, V3(dim == 0 ? 1.f : 0.f, dim == 1 ? 1.f : 0.f, dim == 2 ? 1.f : 0.f));
            V3 lp = -lc, ap = -cross(r_p, lc), ac = cross(r_c, lc);
            float derr = dot(lp, vel_p) + dot(lc, vel_c) + dot(ap, omega_p) + dot(ac, omega_c);
            float err = 0.0f, compliance = P.joint_linear_compliance, damping = 0.0f, alpha_dt = lin_alpha_dt;
            float derr_rel = derr - s.target_vel.get(dim);
            float lo = s.lim_lo.get(dim), up = s.lim_up.get(dim);
            if (e < lo) err = e - lo;
            else if (e > up) err = e - up;
            else {
                float tp = clamp_w(s.target_pos.get(dim), lo, up);
                float ks = s.stiffness.get(dim), kdm = s.damping.get(dim);
                if (ks > 0.0f) {
                    err = e - tp;
                    compliance = 1.0f / ks;
                    damping = kdm;
                } else if (kdm > 0.0f) {
                    compliance = 1.0f / kdm;
                    damping = kdm;
                }
                if (ks > 0.0f || kdm > 0.0f) alpha_dt = compliance / dt;
            }
            if (fabsf(err) > 1e-9f || fabsf(derr_rel) > 1e-9f) {
                float dl = positional_correction(err, derr_rel, bp, bc, lp, lc, ap, ac, compliance, damping, dt, alpha_dt);
                lin_dp += lp * (dl * P.joint_linear_relaxation);
                ang_dp += ap * (dl * P.joint_angular_relaxation);
                lin_dc += lc * (dl * P.joint_linear_relaxation);
                ang_dc += ac * (dl * P.joint_angular_relaxation);
            }
        }
    }

    if (type == JT_FIXED || type == JT_PRISMATIC || type == JT_REVOLUTE || type == JT_D6) {
        const Q4 q_p = X_wp.q;
        Q4 q_c = X_wc.q;
        if (qdot(q_p, q_c) < 0.0f) q_c = qscale(q_c, -1.0f);
        const Q4 rq = qmul(qconj(q_p), q_c);
        const Q4 qtwist = qunit(Q4(rq.x, 0.0f, 0.0f, rq.w));
        const Q4 qswing = qmul(rq, qconj(qtwist));
        const float sn = sqrtf(rq.x * rq.x + rq.w * rq.w);
        const float invs = 1.0f / sn;
        const float invscube = invs * invs * invs;
        float err_0 = 2.0f * asin_w(clamp_w(qtwist.x, -1.0f, 1.0f));
        float err_1 = qswing.y, err_2 = qswing.z;
        Q4 g0(invs - rq.x * rq.x * invscube, 0.0f, 0.0f, -(rq.w * rq.x) * invscube);
        Q4 g1(-rq.w * (rq.w * rq.z + rq.x * rq.y) * invscube, rq.w * invs, -rq.x * invs, rq.x * (rq.w * rq.z + rq.x * rq.y) * invscube);
        Q4 g2(rq.w * (rq.w * rq.y - rq.x * rq.z) * invscube, rq.x * invs, rq.w * invs, rq.x * (rq.z * rq.x - rq.w * rq.y) * invscube);
        g0 = qscale(g0, 2.0f / fabsf(qtwist.w));
        const float swing_sq = qswing.w * qswing.w;
        if (swing_sq + 1.0e-4f < 1.0f) {
            float dd = sqrtf(1.0f - qswing.w * qswing.w);
            float theta = 2.0f * acos_w(clamp_w(qswing.w, -1.0f, 1.0f));
            float scale = theta / dd;
            err_1 *= scale;
            err_2 *= scale;
            g1 = qscale(g1, scale);
            g2 = qscale(g2, scale);
        }
        const AxisSetup s = jc ? load_axis_setup(jc + JC_ANG) : gather_axes(d, ctl, axis_start, target_start, lin_count, ang_count);
        const Q4 qc_inv = qconj(q_c);
#pragma unroll
        for (int dim = 0; dim < 3; ++dim) {
            float e = dim == 0 ? err_0 : (dim == 1 ? err_1 : err_2);
            Q4 grad = dim == 0 ? g0 : (dim == 1 ? g1 : g2);
            Q4 quat_c = qmul(qmul(qscale(q_p, 0.5f), grad), qc_inv);
            V3 ac(quat_c.x, quat_c.y, quat_c.z);
            V3 ap = -ac;
            float derr = dot(ap, omega_p) + dot(ac, omega_c);
            float err = 0.0f, compliance = P.joint_angular_compliance, damping = 0.0f, alpha_dt = ang_alpha_dt;
            float derr_rel = derr - s.target_vel.get(dim) * len(ac);
            float lo = s.lim_lo.get(dim), up = s.lim_up.get(dim);
            if (e < lo) err = e - lo;
            else if (e > up) err = e - up;
            else {
                float tp = clamp_w(s.target_pos.get(dim), lo, up);
                float ks = s.stiffness.get(dim), kdm = s.damping.get(dim);
                if (ks > 0.0f) {
                    err = e - tp;
                    compliance = 1.0f / ks;
                    damping = kdm;
                } else if (kdm > 0.0f) {
                    damping = kdm;
                    compliance = 1.0f / kdm;
                }
                if (ks > 0.0f || kdm > 0.0f) alpha_dt = compliance / dt;
            }
            float dl = angular_correction(err, derr_rel, bp, bc, ap, ac, compliance, damping, dt, alpha_dt) * P.joint_angular_relaxation;
            ang_dp += ap * dl;
            ang_dc += ac * dl;
        }
    }
    out.lin_p = lin_dp;
    out.ang_p = ang_dp;
    out.lin_c = lin_dc;
    out.ang_c = ang_dc;
    return true;
}

// apply_joint_forces for one joint (kernels.py:945-1075): wrench subtracted from the parent / added to the child.
NB2_DEV bool joint_force_wrench(const nb2_model_desc& d, const float* joint_f, int j, int body0, const float* bodies, Deltas& out) {
    const int type = d.joint_type[j];
    if (!d.joint_enabled[j] || type == JT_FIXED || type == JT_ROD) return false;
    const int qd_start = d.joint_qd_start[j];
    const int lin_count = d.joint_dof_dim[2 * j], ang_count = d.joint_dof_dim[2 * j + 1];
    const int ndof = (type == JT_FREE || type == JT_DISTANCE) ? 6 : (type == JT_BALL ? 3 : lin_count + ang_count);
    bool any = false;
    for (int k = 0; k < ndof; ++k) any |= joint_f[qd_start + k] != 0.0f;
    if (!any) return false;  // a zero wrench leaves body_f bit-identical
    const int id_c = d.joint_child[j] - body0;
    const int id_p_raw = d.joint_parent[j];
    const int id_p = id_p_raw >= 0 ? id_p_raw - body0 : -1;
    V3 f_total, t_total;
    if (type == JT_FREE || type == JT_DISTANCE) {
        f_total = V3(joint_f[qd_start], joint_f[qd_start + 1], joint_f[qd_start + 2]);
        t_total = V3(joint_f[qd_start + 3], joint_f[qd_start + 4], joint_f[qd_start + 5]);
        out.lin_p = f_total;
        out.ang_p = t_total;
        out.lin_c = f_total;
        out.ang_c = t_total;
        return true;
    }
    const Xf X_pj = ldx(d.joint_X_p + 7 * j), X_cj = ldx(d.joint_X_c + 7 * j);
    Xf X_wp = X_pj, pose_p = X_pj;
    V3 com_p;
    if (id_p >= 0) {
        pose_p = ldx(bodies + id_p * BR_SIZE + BR_Q);
        X_wp = xmul(pose_p, X_wp);
        com_p = ld3(bodies + id_p * BR_SIZE + BR_COM);
    }
    V3 r_p = X_wp.p - xpoint(pose_p, com_p);
    Xf pose_c = ldx(bodies + id_c * BR_SIZE + BR_Q);
    Xf X_wc = xmul(pose_c, X_cj);
    V3 r_c = X_wc.p - xpoint(pose_c, ld3(bodies + id_c * BR_SIZE + BR_COM));
    if (type == JT_BALL) {
        t_total = V3(joint_f[qd_start], joint_f[qd_start + 1], joint_f[qd_start + 2]);
    } else {
        for (int k = 0; k < 3; ++k)
            if (lin_count > k) f_total += joint_f[qd_start + k] * xvec(X_wp, ld3(d.joint_axis + 3 * (qd_start + k)));
        for (int k = 0; k < 3; ++k)
            if (ang_count > k)
                t_total += joint_f[qd_start + lin_count + k] * xvec(X_wp, ld3(d.joint_axis + 3 * (qd_start + lin_count + k)));
    }
    out.lin_p = f_total;
    out.ang_p = t_total + cross(r_p, f_total);
    out.lin_c = f_total;
    out.ang_c = t_total + cross(r_c, f_total);
    return true;
}

NB2_DEV void store_deltas(float* rec, const Deltas& dl, float active) {
    st3(rec + 0, dl.lin_p);
    st3(rec + 3, dl.ang_p);
    st3(rec + 6, dl.lin_c);
    st3(rec + 9, dl.ang_c);
    rec[12] = active;
}

// apply_body_deltas for one body held in shared memory (kernels.py:864-933), in place.
NB2_DEV void apply_delta(float* rec, V3 dlin, V3 dang, float inv_weight, bool weighted, float dt) {
    const float inv_m = rec[BR_INVM];
    if (inv_m == 0.0f) return;
    const M33 inv_I = ldm(rec + BR_INVI), I = ldm(rec + BR_I);
    const V3 p0 = ld3(rec + BR_Q);
    const Q4 q0(rec[BR_Q + 3], rec[BR_Q + 4], rec[BR_Q + 5], rec[BR_Q + 6]);
    const V3 v0 = ld3(rec + BR_QD), w0 = ld3(rec + BR_QD + 3);
    float weight = 1.0f;
    if (weighted && inv_weight > 0.0f) weight = 1.0f / inv_weight;
    const V3 dp = dlin * (inv_m * weight);
    const V3 dq = dang * weight;
    const V3 wb = qrot_inv(q0, w0);
    const V3 dwb = mv(inv_I, qrot_inv(q0, dq));
    const V3 tb = cross(dwb, mv(I, wb + dwb)) + cross(wb, mv(I, dwb));
    const V3 dw1 = qrot(q0, dwb - mv(mscale(dt, inv_I), tb));
    const V3 h = dw1 * dt;
    Q4 q1 = qadd(q0, qmul(qscale(Q4(h.x, h.y, h.z, 0.0f), 0.5f), q0));
    q1 = qunit(q1);
    const V3 com = ld3(rec + BR_COM);
    const V3 x_com = p0 + qrot(q0, com);
    V3 p1 = x_com + dp * dt;
    p1 -= qrot(q1, com);
    V3 v1 = v0 + dp, w1 = w0 + dw1;
    if (len(v1) < 1e-4f) v1 = V3();
    if (len(w1) < 1e-4f) w1 = V3();
    st3(rec + BR_Q, p1);
    rec[BR_Q + 3] = q1.x; rec[BR_Q + 4] = q1.y; rec[BR_Q + 5] = q1.z; rec[BR_Q + 6] = q1.w;
    st3(rec + BR_QD, v1);
    st3(rec + BR_QD + 3, w1);
}

// ---- 1-D TMA (cp.async.bulk) + mbarrier helpers ------------------------------------------------------------------------
// The CTA's environments own one contiguous run of bodies, so each per-body array of the reference layout (28-byte transforms,
// 24-byte twists, 12-byte centres of mass, 36-byte inertia tensors ...) is ONE contiguous byte range per CTA: a single elected
// thread asks the TMA unit to copy every such run global -> shared (complete_tx on an mbarrier) while the other lanes set up the
// contact and joint tables; at the end of the substep the packed body_q / body_qd runs go back shared -> global as two bulk
// stores.  Bulk copies need 16-byte aligned addresses and sizes, which holds when the CTA's first body index and body count are
// multiples of 4 (4 quadruped envs = 52 bodies): checked per CTA, plain loads / stores otherwise.
NB2_GPU unsigned smem_u32(const void* p) { return static_cast<unsigned>(__cvta_generic_to_shared(p)); }
NB2_GPU void mbar_init(unsigned long long* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
NB2_GPU void mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
NB2_GPU void mbar_wait(unsigned long long* bar, unsigned parity) {
    unsigned done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
}
NB2_GPU void bulk_g2s(void* dst_smem, const void* src_gmem, unsigned bytes, unsigned long long* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst_smem)), "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
NB2_GPU void bulk_s2g(void* dst_gmem, const void* src_smem, unsigned bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst_gmem), "r"(smem_u32(src_smem)), "r"(bytes) : "memory");
}
NB2_GPU void bulk_commit_and_drain() {
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
NB2_GPU void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Shared-memory plan of one CTA (NE environments), in floats.  Identical on host and device.
struct XpbdPlan {
    int bodies, jcache, cpair, ccache, extra, drec, mbar, total;  // offsets of the per-CTA regions
    int rec_cap;                                           // delta records per env; the region doubles as the TMA staging area
};
__host__ __device__ inline XpbdPlan xpbd_plan(int NE, int MB, int MJ, int CC, bool ex, bool joint_cache, int contact_cache = 0) {
    XpbdPlan o;
    auto up4 = [](int x) { return (x + 3) & ~3; };
    o.rec_cap = MB > MJ ? (MB > CC ? MB : CC) : (MJ > CC ? MJ : CC);
    o.bodies = 0;
    o.jcache = up4(o.bodies + NE * MB * BR_SIZE);
    o.cpair = up4(o.jcache + (joint_cache ? NE * MJ * JC_SIZE : 0));
    o.ccache = up4(o.cpair + NE * CC);
    o.extra = up4(o.ccache + NE * contact_cache * CC_SIZE);
    o.drec = up4(o.extra + (ex ? NE * MB * 14 : 0));
    o.mbar = up4(o.drec + NE * o.rec_cap * DR_SIZE);
    o.total = o.mbar + 4;
    return o;
}
// staging layout inside the drec region: nB bodies of the CTA, arrays back to back (each a multiple of 16 bytes when nB % 4 == 0)
enum { ST_Q = 0, ST_QD = 7, ST_COM = 13, ST_INVM = 16, ST_I = 17, ST_INVI = 26, ST_PER_BODY = 35 };

// EX = false: the plain step.  EX = true adds the reporting / post-processing paths of row a17 (restitution, velocity from
// position delta, weighted contact impulses for Contacts.force, joint impulses for State.body_parent_f); it is a second
// instantiation so the plain step pays neither registers nor shared memory for them.
//
// WARPS warps per CTA, each warp = 32/L environments.  All warps of a CTA walk the same code at about the same time, so the
// 6 500-instruction iteration body (far larger than the 32 KB L1.5 instruction cache) is fetched once per CTA instead of once per
// warp; one-warp CTAs each at their own PC were 18 % `stall_no_inst` (profiles/r1f_xpbd_step_kernel.txt).
constexpr int XPBD_MIN_WARPS = 16;  // resident warps per SM the register allocation must allow (16 -> 128 registers)
template <int L, bool EX, int WARPS>
__global__ void __launch_bounds__(32 * WARPS, (WARPS >= XPBD_MIN_WARPS ? 1 : XPBD_MIN_WARPS / WARPS))
xpbd_step_kernel(DevModel M, nb2_xpbd_params P, nb2_state_view sin, nb2_state_view sout, nb2_control_view ctl, int use_contacts_flags,
                 float dt, bool joint_cache, int contact_cap, int contact_cache) {
    const int use_contacts = use_contacts_flags & NB2_XPBD_USE_CONTACTS;
    const bool want_cimp = EX && use_contacts && (use_contacts_flags & NB2_XPBD_CONTACT_IMPULSE);
    const bool want_jimp = EX && sout.body_parent_f != nullptr;
    const bool want_init = EX && (P.enable_restitution || P.compute_body_velocity_from_position_delta);
    constexpr int G = 32 / L;
    constexpr int NE = G * WARPS;
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / L, l = lane % L;
    const int slot = warp * G + grp;  // environment slot inside the CTA
    const int env0 = blockIdx.x * NE;
    const int env = env0 + slot;
    const bool live = env < M.env_count;
    const nb2_model_desc& d = M.d;
    const XpbdPlan plan = xpbd_plan(NE, M.max_env_bodies, M.max_env_joints, contact_cap, EX, joint_cache, contact_cache);
    float* ccache = smem + plan.ccache + slot * contact_cache * CC_SIZE;  // first `contact_cache` contacts of the environment
    float* bodies = smem + plan.bodies + slot * M.max_env_bodies * BR_SIZE;
    float* drec = smem + plan.drec + slot * plan.rec_cap * DR_SIZE;
    int* cpair = reinterpret_cast<int*>(smem + plan.cpair) + slot * contact_cap;
    float* init_qd = smem + plan.extra + slot * M.max_env_bodies * 14;  // EX only: state_in poses + twists (13/body)
    float* bcnt = init_qd + M.max_env_bodies * 13;                       // EX only: active contacts per body
    float* jcache = joint_cache ? smem + plan.jcache + slot * M.max_env_joints * JC_SIZE : nullptr;
    float* stage = smem + plan.drec;  // CTA-wide staging area of the bulk copies (the delta records are not live then)
    unsigned long long* mbar = reinterpret_cast<unsigned long long*>(smem + plan.mbar);

    int b0 = 0, nb = 0, j0 = 0, nj = 0, slot0 = 0, nc = 0;
    if (live) {
        b0 = M.env_body_start[env];
        nb = M.env_body_start[env + 1] - b0;
        j0 = M.env_joint_start[env];
        nj = M.env_joint_start[env + 1] - j0;
        slot0 = M.env_slot_start[env];
        nc = use_contacts ? min(M.env_contact_count[env], contact_cap) : 0;
    }
    // ---- body state + constants -> shared memory ------------------------------------------------------------------------------
    // CTA-uniform decision: the CTA's body run [cb0, cb0 + cnb) must be 16-byte aligned in every array it is copied from / to
    const int env_last = min(env0 + NE, M.env_count);
    const int cb0 = M.env_body_start[env0], cnb = M.env_body_start[env_last] - cb0;
    bool tma = cnb > 0 && (cb0 & 3) == 0 && (cnb & 3) == 0 && cnb * ST_PER_BODY <= NE * plan.rec_cap * DR_SIZE;
    if (tma) {
        const uintptr_t a = reinterpret_cast<uintptr_t>(sin.body_q) | reinterpret_cast<uintptr_t>(sin.body_qd) |
                            reinterpret_cast<uintptr_t>(sout.body_q) | reinterpret_cast<uintptr_t>(sout.body_qd) |
                            reinterpret_cast<uintptr_t>(d.body_com) | reinterpret_cast<uintptr_t>(d.body_inv_mass) |
                            reinterpret_cast<uintptr_t>(d.body_inertia) | reinterpret_cast<uintptr_t>(d.body_inv_inertia);
        tma = (a & 15) == 0;
    }
    if (tma) {
        if (threadIdx.x == 0) mbar_init(mbar, 1);
        __syncthreads();
        if (threadIdx.x == 0) {
            mbar_expect_tx(mbar, unsigned(cnb) * ST_PER_BODY * 4u);
            bulk_g2s(stage + ST_Q * cnb, sin.body_q + 7 * size_t(cb0), unsigned(cnb) * 28u, mbar);
            bulk_g2s(stage + ST_QD * cnb, sin.body_qd + 6 * size_t(cb0), unsigned(cnb) * 24u, mbar);
            bulk_g2s(stage + ST_COM * cnb, d.body_com + 3 * size_t(cb0), unsigned(cnb) * 12u, mbar);
            bulk_g2s(stage + ST_INVM * cnb, d.body_inv_mass + size_t(cb0), unsigned(cnb) * 4u, mbar);
            bulk_g2s(stage + ST_I * cnb, d.body_inertia + 9 * size_t(cb0), unsigned(cnb) * 36u, mbar);
            bulk_g2s(stage + ST_INVI * cnb, d.body_inv_inertia + 9 * size_t(cb0), unsigned(cnb) * 36u, mbar);
        }
    }
    // (while the copies are in flight) contact -> body incidence and the joint cache
    for (int c = l; c < nc; c += L) {
        const size_t T = size_t(M.slot_total);
        int ba = __float_as_int(M.cb[CF_BODY_A * T + slot0 + c]), bb = __float_as_int(M.cb[CF_BODY_B * T + slot0 + c]);
        // packed incidence: 15-bit body index + 1 per side (0 = the static world) and the body's KINEMATIC flag, so the
        // iteration loop never goes back to global memory for them
        const unsigned ka = ba >= 0 && (d.body_flags[b0 + ba] & BODY_KINEMATIC) != 0, kb = bb >= 0 && (d.body_flags[b0 + bb] & BODY_KINEMATIC) != 0;
        cpair[c] = int(unsigned(ba + 1) | (ka << 15) | (unsigned(bb + 1) << 16) | (kb << 31));
        if (c < contact_cache) {
            const int s = slot0 + c;
            float* cc = ccache + c * CC_SIZE;
            const V3 p0(M.cb[CF_P0X * T + s], M.cb[CF_P0Y * T + s], M.cb[CF_P0Z * T + s]);
            const V3 p1(M.cb[CF_P1X * T + s], M.cb[CF_P1Y * T + s], M.cb[CF_P1Z * T + s]);
            const V3 o0(M.cb[CF_O0X * T + s], M.cb[CF_O0Y * T + s], M.cb[CF_O0Z * T + s]);
            const V3 o1(M.cb[CF_O1X * T + s], M.cb[CF_O1Y * T + s], M.cb[CF_O1Z * T + s]);
            st3(cc + CC_P0, p0);
            st3(cc + CC_P1, p1);
            st3(cc + CC_N, V3(M.cb[CF_NX * T + s], M.cb[CF_NY * T + s], M.cb[CF_NZ * T + s]));
            cc[CC_MSUM] = M.cb[CF_MARGIN0 * T + s] + M.cb[CF_MARGIN1 * T + s];
            cc[CC_MU] = M.cb[CF_MU * T + s];
            cc[CC_MUT] = M.cb[CF_MU_TORSIONAL * T + s];
            cc[CC_MUR] = M.cb[CF_MU_ROLLING * T + s];
            st3(cc + CC_Q0, p0 + o0);
            st3(cc + CC_Q1, p1 + o1);
        }
        if (want_cimp)
#pragma unroll
            for (int k = 0; k < 6; ++k) M.contact_impulse[k * T + slot0 + c] = 0.0f;
    }
    if (jcache)
        for (int j = l; j < nj; j += L) {
            const int gj = j0 + j;
            float* jc = jcache + j * JC_SIZE;
            const int lin_count = d.joint_dof_dim[2 * gj], ang_count = d.joint_dof_dim[2 * gj + 1];
            const int axis_start = d.joint_qd_start[gj], target_start = d.joint_target_q_start[gj];
            stx(jc + JC_XP, ldx(d.joint_X_p + 7 * gj));
            stx(jc + JC_XC, ldx(d.joint_X_c + 7 * gj));
            store_axis_setup(jc + JC_ANG, gather_axes(d, ctl, axis_start, target_start, lin_count, ang_count));
            jc[JC_HDR] = __int_as_float(d.joint_type[gj] | (d.joint_enabled[gj] ? 16 : 0) | (lin_count << 8) | (ang_count << 12));
            jc[JC_CHILD] = __int_as_float(d.joint_child[gj]);
            jc[JC_PARENT] = __int_as_float(d.joint_parent[gj]);
            jc[JC_AXIS] = __int_as_float(axis_start);
            jc[JC_TARGET] = __int_as_float(target_start);
        }
    if (tma) mbar_wait(mbar, 0);
    for (int b = l; b < nb; b += L) {
        const int gb = b0 + b;
        float* rec = bodies + b * BR_SIZE;
        const bool kin = (d.body_flags[gb] & BODY_KINEMATIC) != 0;  // _update_effective_inv_mass_inertia (solver.py:173-187)
        if (tma) {
            const int sb = gb - cb0;
#pragma unroll
            for (int k = 0; k < 7; ++k) rec[BR_Q + k] = stage[ST_Q * cnb + 7 * sb + k];
#pragma unroll
            for (int k = 0; k < 6; ++k) rec[BR_QD + k] = stage[ST_QD * cnb + 6 * sb + k];
#pragma unroll
            for (int k = 0; k < 3; ++k) rec[BR_COM + k] = stage[ST_COM * cnb + 3 * sb + k];
            rec[BR_INVM] = kin ? 0.0f : stage[ST_INVM * cnb + sb];
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                rec[BR_INVI + k] = kin ? 0.0f : stage[ST_INVI * cnb + 9 * sb + k];
                rec[BR_I + k] = stage[ST_I * cnb + 9 * sb + k];
            }
        } else {
#pragma unroll
            for (int k = 0; k < 7; ++k) rec[BR_Q + k] = sin.body_q[7 * gb + k];
#pragma unroll
            for (int k = 0; k < 6; ++k) rec[BR_QD + k] = sin.body_qd[6 * gb + k];
#pragma unroll
            for (int k = 0; k < 3; ++k) rec[BR_COM + k] = d.body_com[3 * gb + k];
            rec[BR_INVM] = kin ? 0.0f : d.body_inv_mass[gb];
#pragma unroll
            for (int k = 0; k < 9; ++k) {
                rec[BR_INVI + k] = kin ? 0.0f : d.body_inv_inertia[9 * gb + k];
                rec[BR_I + k] = d.body_inertia[9 * gb + k];
            }
        }
    }
    if (want_init)
        for (int b = l; b < nb; b += L)
#pragma unroll
            for (int k = 0; k < 13; ++k) init_qd[b * 13 + k] = bodies[b * BR_SIZE + BR_Q + k];  // q (7) then qd (6) are adjacent
    if (tma) __syncthreads();  // every warp has unpacked its bodies: the staging area becomes the delta records
    else __syncwarp();
    // ---- contact -> body incidence as two bit masks per body lane (contact c touches this body on side A / side B) --------------
    // Contact order is the summation order; a mask walk visits exactly the incident records in that order instead of rescanning
    // all nc contacts per body per iteration.  One body per lane and <= 64 contacts; larger environments use the scan.
    const bool use_masks = nb <= L && nc <= 64;
    unsigned long long mask_a = 0ull, mask_b = 0ull;
    if (use_masks && l < nb)
        for (int c = 0; c < nc; ++c) {
            const int pr = cpair[c];
            const int ba = int(unsigned(pr) & 0x7fffu) - 1, bb = int((unsigned(pr) >> 16) & 0x7fffu) - 1;
            if (ba == bb) continue;  // the contact pass writes an inactive record
            if (ba == l) mask_a |= 1ull << c;
            if (bb == l) mask_b |= 1ull << c;
        }
    // ---- apply_joint_forces: per-joint wrenches, then ordered per-body accumulation into a body_f copy ----
    for (int j = l; j < nj; j += L) {
        Deltas w;
        bool act = joint_force_wrench(d, ctl.joint_f, j0 + j, b0, bodies, w);
        if (!act) w = Deltas();
        store_deltas(drec + j * DR_SIZE, w, act ? 1.0f : 0.0f);
        if (want_jimp) {  // child-side wrench * dt opens the joint's impulse accumulator (kernels.py:1018-1019, 1074-1075)
            float* ji = M.joint_impulse + 6 * size_t(j0 + j);
            const V3 a = V3() + w.lin_c * dt, t = V3() + w.ang_c * dt;
            st3(ji, a);
            st3(ji + 3, t);
        }
    }
    __syncwarp();
    // ---- integrate_bodies (solver.py:64-107) ----------------------------------------------------
    for (int b = l; b < nb; b += L) {
        const int gb = b0 + b;
        float* rec = bodies + b * BR_SIZE;
        V3 f0 = ld3(sin.body_f + 6 * gb), t0 = ld3(sin.body_f + 6 * gb + 3);
        for (int k = M.body_joint_start[gb]; k < M.body_joint_start[gb + 1]; ++k) {
            const int e = M.body_joint_entry[k];
            const float* r = drec + (e >> 1) * DR_SIZE;
            if (r[12] != 0.0f) {
                if (e & 1) { f0 += ld3(r + 6); t0 += ld3(r + 9); }
                else { f0 -= ld3(r + 0); t0 -= ld3(r + 3); }
            }
        }
        if ((d.body_flags[gb] & BODY_KINEMATIC) != 0) continue;  // kinematic bodies pass through (solver.py:132-139)
        const V3 x0 = ld3(rec + BR_Q);
        const Q4 r0(rec[BR_Q + 3], rec[BR_Q + 4], rec[BR_Q + 5], rec[BR_Q + 6]);
        const V3 v0 = ld3(rec + BR_QD), w0 = ld3(rec + BR_QD + 3);
        const V3 com = ld3(rec + BR_COM);
        const float inv_mass = rec[BR_INVM];  // not kinematic here: the effective value is the model's
        const M33 inertia = ldm(rec + BR_I);
        const M33 inv_inertia = ldm(rec + BR_INVI);
        int wi = d.body_world[gb];
        if (wi < 0) wi += d.gravity_count;
        const V3 g = ld3(d.gravity + 3 * wi);
        const V3 x_com = x0 + qrot(r0, com);
        const V3 v1 = v0 + (f0 * inv_mass + g * (inv_mass != 0.0f ? 1.0f : 0.0f)) * dt;
        const V3 x1 = x_com + v1 * dt;
        const V3 wb = qrot_inv(r0, w0);
        const V3 tb = qrot_inv(r0, t0) - cross(wb, mv(inertia, wb));
        V3 w1 = qrot(r0, wb + mv(inv_inertia, tb) * dt);
        const Q4 r1 = qunit(qadd(r0, qscale(qscale(qmul(Q4(w1.x, w1.y, w1.z, 0.0f), r0), 0.5f), dt)));
        w1 *= 1.0f - P.angular_damping * dt;
        st3(rec + BR_Q, x1 - qrot(r1, com));
        rec[BR_Q + 3] = r1.x; rec[BR_Q + 4] = r1.y; rec[BR_Q + 5] = r1.z; rec[BR_Q + 6] = r1.w;
        st3(rec + BR_QD, v1);
        st3(rec + BR_QD + 3, w1);
    }
    __syncwarp();
    // ---- Jacobi iterations ---------------------------------------------------------------------------
    const size_t T = size_t(M.slot_total);
    const float* cb = M.cb;
    // compliance / dt of the rows that use the solver-wide compliance (limit rows, locked axes): the same for every joint, row and
    // iteration, so divided once here instead of in every row of every iteration
    const float lin_alpha_dt = P.joint_linear_compliance / dt, ang_alpha_dt = P.joint_angular_compliance / dt;
    for (int it = 0; it < P.iterations; ++it) {
        // CTA barriers are not needed for correctness (a warp owns its environments); they keep the CTA's warps on the same
        // stretch of code so that the instruction stream is fetched once per CTA (see the kernel comment).  One per iteration: 147.8 us,
        // against 154.4 us without barriers and 151.9 us with one at every phase boundary (DESIGN.md section 3.1)
        if (WARPS > 1) __syncthreads();
        if (use_contacts) {
            // ---- [iteration] solve_body_contact_positions (kernels.py:2164-2399)
            for (int c = l; c < nc; c += L) {
                const int s = slot0 + c;
                const int pr = cpair[c];
                const int ba = int(unsigned(pr) & 0x7fffu) - 1, bb = int((unsigned(pr) >> 16) & 0x7fffu) - 1;
                Deltas dl;
                float active = 0.0f;
                if (ba != bb) {
                    // A side never consumed by a body (static world) and not reported: its arithmetic is skipped.  Identity
                    // transform and zero centre of mass reduce xpoint(X, p) to (+0) + p and r to the contact point itself.
                    const bool need_a = ba >= 0 || want_cimp, need_b = bb >= 0 || want_cimp;
                    BodyView A = ba >= 0 ? load_body(bodies + ba * BR_SIZE) : static_body();
                    BodyView B = bb >= 0 ? load_body(bodies + bb * BR_SIZE) : static_body();
                    const bool cached = c < contact_cache;
                    const float* cc = ccache + c * CC_SIZE;
                    const V3 p0 = cached ? ld3(cc + CC_P0) : V3(cb[CF_P0X * T + s], cb[CF_P0Y * T + s], cb[CF_P0Z * T + s]);
                    const V3 p1 = cached ? ld3(cc + CC_P1) : V3(cb[CF_P1X * T + s], cb[CF_P1Y * T + s], cb[CF_P1Z * T + s]);
                    const V3 n = cached ? ld3(cc + CC_N) : V3(cb[CF_NX * T + s], cb[CF_NY * T + s], cb[CF_NZ * T + s]);
                    V3 bx_a = ba >= 0 ? xpoint(A.X, p0) : V3() + p0, bx_b = bb >= 0 ? xpoint(B.X, p1) : V3() + p1;
                    const float dpen = dot(n, bx_b - bx_a) - (cached ? cc[CC_MSUM] : cb[CF_MARGIN0 * T + s] + cb[CF_MARGIN1 * T + s]);
                    if (dpen < 0.0f) {
                        active = 1.0f;
                        const float mu = cached ? cc[CC_MU] : cb[CF_MU * T + s], mu_t = cached ? cc[CC_MUT] : cb[CF_MU_TORSIONAL * T + s],
                                    mu_r = cached ? cc[CC_MUR] : cb[CF_MU_ROLLING * T + s];
                        const V3 wcom_a = ba >= 0 ? xpoint(A.X, A.com) : V3(), wcom_b = bb >= 0 ? xpoint(B.X, B.com) : V3();
                        V3 r_a = bx_a - wcom_a, r_b = bx_b - wcom_b;
                        V3 ang_a, ang_b;
                        if (need_a) ang_a = -cross(r_a, n);
                        if (need_b) ang_b = cross(r_b, n);
                        const float lambda_n = contact_delta(dpen, A, B, -n, n, ang_a, ang_b, P.rigid_contact_relaxation, dt);
                        V3 lin_da, lin_db, ang_da, ang_db;
                        if (need_a) { lin_da = -n * lambda_n; ang_da = ang_a * lambda_n; }
                        if (need_b) { lin_db = n * lambda_n; ang_db = ang_b * lambda_n; }
                        if (mu > 0.0f) {
                            V3 q0, q1;  // contact_surface_point: point + offset
                            if (cached) {
                                q0 = ld3(cc + CC_Q0);
                                q1 = ld3(cc + CC_Q1);
                            } else {
                                q0 = p0 + V3(cb[CF_O0X * T + s], cb[CF_O0Y * T + s], cb[CF_O0Z * T + s]);
                                q1 = p1 + V3(cb[CF_O1X * T + s], cb[CF_O1Y * T + s], cb[CF_O1Z * T + s]);
                            }
                            bx_a = ba >= 0 ? xpoint(A.X, q0) : V3() + q0;
                            bx_b = bb >= 0 ? xpoint(B.X, q1) : V3() + q1;
                            V3 delta = bx_b - bx_a;
                            V3 fd = delta - dot(n, delta) * n;
                            r_a = bx_a - wcom_a;
                            r_b = bx_b - wcom_b;
                            V3 rel_v_kin;
                            if (unsigned(pr) & 0x8000u) {  // body A is kinematic
                                V3 v_a = cross(A.w, r_a) + A.v;
                                rel_v_kin = rel_v_kin - (v_a - dot(n, v_a) * n);
                            }
                            if (unsigned(pr) & 0x80000000u) {  // body B is kinematic
                                V3 v_b = cross(B.w, r_b) + B.v;
                                rel_v_kin = rel_v_kin + (v_b - dot(n, v_b) * n);
                            }
                            fd += rel_v_kin * dt;
                            V3 perp = unit(fd);
                            if (need_a) ang_a = -cross(r_a, perp);
                            if (need_b) ang_b = cross(r_b, perp);
                            float err = len(fd);
                            if (err > 0.0f) {
                                float lambda_fr = contact_delta(err, A, B, -perp, perp, ang_a, ang_b, P.rigid_contact_relaxation, dt);
                                lambda_fr = fmax_w(lambda_fr, -lambda_n * mu);
                                if (need_a) { lin_da -= perp * lambda_fr; ang_da += ang_a * lambda_fr; }
                                if (need_b) { lin_db += perp * lambda_fr; ang_db += ang_b * lambda_fr; }
                            }
                        }
                        V3 dom = B.w - A.w;
                        if (mu_t > 0.0f) {
                            float err = dot(dom, n) * dt;
                            if (fabsf(err) > 0.0f) {
                                float lt = contact_delta(err, A, B, V3(), V3(), -n, n, P.rigid_contact_relaxation, dt);
                                lt = clamp_w(lt, -lambda_n * mu_t, lambda_n * mu_t);
                                if (need_a) ang_da -= n * lt;
                                if (need_b) ang_db += n * lt;
                            }
                        }
                        if (mu_r > 0.0f) {
                            dom -= dot(n, dom) * n;
                            float err = len(dom) * dt;
                            if (err > 0.0f) {
                                V3 rn = unit(dom);
                                float lr = contact_delta(err, A, B, V3(), V3(), -rn, rn, P.rigid_contact_relaxation, dt);
                                lr = fmax_w(lr, -lambda_n * mu_r);
                                if (need_a) ang_da -= rn * lr;
                                if (need_b) ang_db += rn * lr;
                            }
                        }
                        dl.lin_p = lin_da;
                        dl.ang_p = ang_da;
                        dl.lin_c = lin_db;
                        dl.ang_c = ang_db;
                    }
                }
                store_deltas(drec + c * DR_SIZE, dl, active);
            }
            __syncwarp();
            // ---- [iteration] ordered per-body sum (contact order; side A before side B) + weighted apply
            for (int b = l; b < nb; b += L) {
                V3 dlin, dang;
                float cnt = 0.0f;
                if (use_masks) {
                    unsigned long long m = mask_a | mask_b;
                    while (m) {
                        const int c = __ffsll((long long)m) - 1;
                        m &= m - 1;
                        const float* r = drec + c * DR_SIZE;
                        if (r[12] == 0.0f) continue;
                        if ((mask_a >> c) & 1ull) { dlin += ld3(r + 0); dang += ld3(r + 3); cnt += 1.0f; }
                        if ((mask_b >> c) & 1ull) { dlin += ld3(r + 6); dang += ld3(r + 9); cnt += 1.0f; }
                    }
                } else {
                    for (int c = 0; c < nc; ++c) {
                        const int pr = cpair[c];
                        const int ba = int(unsigned(pr) & 0x7fffu) - 1, bb = int((unsigned(pr) >> 16) & 0x7fffu) - 1;
                        if (ba != b && bb != b) continue;
                        const float* r = drec + c * DR_SIZE;
                        if (r[12] == 0.0f) continue;
                        if (ba == b) { dlin += ld3(r + 0); dang += ld3(r + 3); cnt += 1.0f; }
                        if (bb == b) { dlin += ld3(r + 6); dang += ld3(r + 9); cnt += 1.0f; }
                    }
                }
                apply_delta(bodies + b * BR_SIZE, dlin, dang, cnt, P.rigid_contact_con_weighting != 0, dt);
                if (want_cimp) bcnt[b] = cnt;
            }
            __syncwarp();
            if (want_cimp) {  // accumulate_weighted_contact_impulse (kernels.py:2402-2461)
                for (int c = l; c < nc; c += L) {
                    const float* r = drec + c * DR_SIZE;
                    if (r[12] == 0.0f) continue;  // inactive this iteration: the reference adds an exact zero
                    const int pr = cpair[c];
                    const int ba = int(unsigned(pr) & 0x7fffu) - 1, bb = int((unsigned(pr) >> 16) & 0x7fffu) - 1;
                    float weight = 1.0f;
                    if (P.rigid_contact_con_weighting) {
                        const float n_a = ba >= 0 ? bcnt[ba] : 0.0f, n_b = bb >= 0 ? bcnt[bb] : 0.0f;
                        const float n_sum = n_a + n_b;
                        if (n_sum > 0.0f) {
                            if (n_a == 0.0f) weight = 1.0f / n_b;
                            else if (n_b == 0.0f) weight = 1.0f / n_a;
                            else weight = 2.0f / n_sum;
                        }
                    }
                    float* ci = M.contact_impulse + slot0 + c;
#pragma unroll
                    for (int k = 0; k < 6; ++k) ci[k * T] = ci[k * T] + r[k] * weight;  // (lin_delta_a, ang_delta_a) * weight
                }
                __syncwarp();
            }
        }
        if (d.joint_count > 0) {
            // ---- [iteration] solve_body_joints (kernels.py:1513-2044) + ordered per-body apply
            for (int j = l; j < nj; j += L) {
                Deltas dl;
                bool act = solve_joint(d, ctl, P, j0 + j, b0, bodies, jcache ? jcache + j * JC_SIZE : nullptr, dt, lin_alpha_dt,
                                       ang_alpha_dt, dl);
                if (!act) dl = Deltas();
                store_deltas(drec + j * DR_SIZE, dl, act ? 1.0f : 0.0f);
                if (want_jimp && act) {  // kernels.py:2043-2044
                    float* ji = M.joint_impulse + 6 * size_t(j0 + j);
                    st3(ji, ld3(ji) + dl.lin_c);
                    st3(ji + 3, ld3(ji + 3) + dl.ang_c);
                }
            }
            __syncwarp();
            for (int b = l; b < nb; b += L) {
                const int gb = b0 + b;
                V3 dlin, dang;
                for (int k = M.body_joint_start[gb]; k < M.body_joint_start[gb + 1]; ++k) {
                    const int e = M.body_joint_entry[k];
                    const float* r = drec + (e >> 1) * DR_SIZE;
                    if (r[12] == 0.0f) continue;
                    if (e & 1) { dlin += ld3(r + 6); dang += ld3(r + 9); }
                    else { dlin += ld3(r + 0); dang += ld3(r + 3); }
                }
                apply_delta(bodies + b * BR_SIZE, dlin, dang, 0.0f, false, dt);
            }
            __syncwarp();
        }
    }
    if (EX) {
        // ---- State.body_parent_f (convert_joint_impulse_to_parent_f, kernels.py:2497-2544): joints in index order per child ----
        if (sout.body_parent_f != nullptr) {
            __syncwarp();
            const float inv_dt = 1.0f / dt;
            for (int b = l; b < nb; b += L) {
                const int gb = b0 + b;
                V3 f, t;
                for (int k = M.body_joint_start[gb]; k < M.body_joint_start[gb + 1]; ++k) {
                    const int e = M.body_joint_entry[k];
                    if (!(e & 1)) continue;
                    const int gj = j0 + (e >> 1);
                    if (!d.joint_enabled[gj] || d.joint_type[gj] == JT_FREE) continue;
                    const float* ji = M.joint_impulse + 6 * size_t(gj);
                    f += ld3(ji) * inv_dt;
                    t += ld3(ji + 3) * inv_dt;
                }
                st3(sout.body_parent_f + 6 * gb, f);
                st3(sout.body_parent_f + 6 * gb + 3, t);
            }
        }
        // ---- update_body_velocities (kernels.py:2547-2579); kinematic bodies keep their input state (copy_kinematic) -----------
        if (P.compute_body_velocity_from_position_delta) {
            for (int b = l; b < nb; b += L) {
                if ((d.body_flags[b0 + b] & BODY_KINEMATIC) != 0) continue;
                float* rec = bodies + b * BR_SIZE;
                const Xf pose = ldx(rec + BR_Q), prev = ldx(init_qd + b * 13);
                const V3 com = ld3(rec + BR_COM);
                const V3 x_com = pose.p + qrot(pose.q, com), x_prev = prev.p + qrot(prev.q, com);
                const V3 v = (x_com - x_prev) / dt;
                const Q4 dq = qmul(pose.q, qconj(prev.q));
                V3 omega = (2.0f / dt) * V3(dq.x, dq.y, dq.z);
                if (dq.w < 0.0f) omega = -omega;
                st3(rec + BR_QD, v);
                st3(rec + BR_QD + 3, omega);
            }
            __syncwarp();
        }
        // ---- apply_rigid_restitution (kernels.py:2582-2728) + apply_body_delta_velocities (:936-942) ------------------------------
        if (P.enable_restitution && use_contacts) {
            for (int c = l; c < nc; c += L) {
                const int s = slot0 + c;
                const int pr = cpair[c];
                const int ba = int(unsigned(pr) & 0x7fffu) - 1, bb = int((unsigned(pr) >> 16) & 0x7fffu) - 1;
                Deltas dl;
                float active = 0.0f;
                if (ba != bb) {
                    const int sa = __float_as_int(cb[CF_SHAPE0 * T + s]), sb = __float_as_int(cb[CF_SHAPE1 * T + s]);
                    float restitution = 0.0f;
                    restitution += d.shape_material_restitution[sa];
                    restitution += d.shape_material_restitution[sb];
                    restitution /= 2.0f;
                    const float* ra_rec = ba >= 0 ? bodies + ba * BR_SIZE : nullptr;
                    const float* rb_rec = bb >= 0 ? bodies + bb * BR_SIZE : nullptr;
                    const Xf Xa = ba >= 0 ? ldx(init_qd + ba * 13) : Xf(), Xb = bb >= 0 ? ldx(init_qd + bb * 13) : Xf();
                    const V3 com_a = ba >= 0 ? ld3(ra_rec + BR_COM) : V3(), com_b = bb >= 0 ? ld3(rb_rec + BR_COM) : V3();
                    const V3 p0(cb[CF_P0X * T + s], cb[CF_P0Y * T + s], cb[CF_P0Z * T + s]);
                    const V3 p1(cb[CF_P1X * T + s], cb[CF_P1Y * T + s], cb[CF_P1Z * T + s]);
                    const V3 o0(cb[CF_O0X * T + s], cb[CF_O0Y * T + s], cb[CF_O0Z * T + s]);
                    const V3 o1(cb[CF_O1X * T + s], cb[CF_O1Y * T + s], cb[CF_O1Z * T + s]);
                    const V3 n(cb[CF_NX * T + s], cb[CF_NY * T + s], cb[CF_NZ * T + s]);
                    const V3 bx_a = xpoint(Xa, p0 + o0), bx_b = xpoint(Xb, p1 + o1);  // contact_surface_point
                    if (dot(n, bx_b - bx_a) < 0.0f) {
                        const V3 r_a = bx_a - xpoint(Xa, com_a), r_b = bx_b - xpoint(Xb, com_b);
                        V3 v_a, v_b, v_a_new, v_b_new, rxn_a, rxn_b;
                        float inv_mass = 0.0f, m_inv_a = 0.0f, m_inv_b = 0.0f;
                        M33 I_inv_a = m33_zero(), I_inv_b = m33_zero();
                        if (ba >= 0) {
                            int wi = d.body_world[b0 + ba];
                            if (wi < 0) wi += d.gravity_count;
                            m_inv_a = ra_rec[BR_INVM];
                            I_inv_a = ldm(ra_rec + BR_INVI);
                            v_a = (cross(ld3(init_qd + ba * 13 + 10), r_a) + ld3(init_qd + ba * 13 + 7)) + ld3(d.gravity + 3 * wi) * dt;
                            v_a_new = cross(ld3(ra_rec + BR_QD + 3), r_a) + ld3(ra_rec + BR_QD);
                            rxn_a = qrot_inv(Xa.q, cross(r_a, n));
                            inv_mass += m_inv_a + dot(rxn_a, mv(I_inv_a, rxn_a));
                        }
                        if (bb >= 0) {
                            int wi = d.body_world[b0 + bb];
                            if (wi < 0) wi += d.gravity_count;
                            m_inv_b = rb_rec[BR_INVM];
                            I_inv_b = ldm(rb_rec + BR_INVI);
                            v_b = (cross(ld3(init_qd + bb * 13 + 10), r_b) + ld3(init_qd + bb * 13 + 7)) + ld3(d.gravity + 3 * wi) * dt;
                            v_b_new = cross(ld3(rb_rec + BR_QD + 3), r_b) + ld3(rb_rec + BR_QD);
                            rxn_b = qrot_inv(Xb.q, cross(r_b, n));
                            inv_mass += m_inv_b + dot(rxn_b, mv(I_inv_b, rxn_b));
                        }
                        const float rel_old = dot(n, v_b - v_a), rel_new = dot(n, v_b_new - v_a_new);
                        if (inv_mass != 0.0f && rel_old < 0.0f) {
                            const float dv = (-rel_new - restitution * rel_old) / inv_mass;
                            active = 1.0f;
                            if (ba >= 0) {
                                const float dv_a = -dv;
                                dl.lin_p = n * m_inv_a * dv_a;
                                dl.ang_p = qrot(Xa.q, mv(I_inv_a, rxn_a) * dv_a);
                            }
                            if (bb >= 0) {
                                dl.lin_c = n * m_inv_b * dv;
                                dl.ang_c = qrot(Xb.q, mv(I_inv_b, rxn_b) * dv);
                            }
                        }
                    }
                }
                store_deltas(drec + c * DR_SIZE, dl, active);
            }
            __syncwarp();
            for (int b = l; b < nb; b += L) {
                if ((d.body_flags[b0 + b] & BODY_KINEMATIC) != 0) continue;
                V3 dlin, dang;
                for (int c = 0; c < nc; ++c) {
                    const int pr = cpair[c];
                    const int ba = int(unsigned(pr) & 0x7fffu) - 1, bb = int((unsigned(pr) >> 16) & 0x7fffu) - 1;
                    if (ba != b && bb != b) continue;
                    const float* r = drec + c * DR_SIZE;
                    if (r[12] == 0.0f) continue;
                    if (ba == b) { dlin += ld3(r + 0); dang += ld3(r + 3); }
                    if (bb == b) { dlin += ld3(r + 6); dang += ld3(r + 9); }
                }
                float* rec = bodies + b * BR_SIZE;
                st3(rec + BR_QD, ld3(rec + BR_QD) + dlin);
                st3(rec + BR_QD + 3, ld3(rec + BR_QD + 3) + dang);
            }
            __syncwarp();
        }
    }
    // ---- write back -------------------------------------------------------------------------------------
    if (tma) {
        // pack the CTA's body_q / body_qd runs in the reference's AoS layout, then two bulk stores shared -> global
        __syncthreads();  // all warps are done with their delta records: the region is the staging area again
        for (int b = l; b < nb; b += L) {
            const int sb = b0 + b - cb0;
            const float* rec = bodies + b * BR_SIZE;
#pragma unroll
            for (int k = 0; k < 7; ++k) stage[ST_Q * cnb + 7 * sb + k] = rec[BR_Q + k];
#pragma unroll
            for (int k = 0; k < 6; ++k) stage[ST_QD * cnb + 6 * sb + k] = rec[BR_QD + k];
        }
        fence_async_smem();  // generic-proxy writes -> visible to the async proxy (TMA)
        __syncthreads();
        if (threadIdx.x == 0) {
            bulk_s2g(sout.body_q + 7 * size_t(cb0), stage + ST_Q * cnb, unsigned(cnb) * 28u);
            bulk_s2g(sout.body_qd + 6 * size_t(cb0), stage + ST_QD * cnb, unsigned(cnb) * 24u);
            bulk_commit_and_drain();  // shared memory must stay alive until the TMA unit has read it
        }
        return;
    }
    for (int b = l; b < nb; b += L) {
        const int gb = b0 + b;
        const float* rec = bodies + b * BR_SIZE;
#pragma unroll
        for (int k = 0; k < 7; ++k) sout.body_q[7 * gb + k] = rec[BR_Q + k];
#pragma unroll
        for (int k = 0; k < 6; ++k) sout.body_qd[6 * gb + k] = rec[BR_QD + k];
    }
}

// SolverXPBD.update_contacts (solver_xpbd.py:864-925): force[i] = weighted impulse of exported contact i / dt
__global__ void __launch_bounds__(128) xpbd_update_contacts_kernel(DevModel M, nb2_contacts_view out, float inv_dt) {
    const int env = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5);
    if (env >= M.env_count) return;
    const int lane = threadIdx.x & 31;
    const int n = M.env_contact_count[env], base = M.env_contact_offset[env], slot0 = M.env_slot_start[env];
    const size_t T = size_t(M.slot_total);
    for (int c = lane; c < n; c += 32) {
        int o = base + c;
        if (o >= out.rigid_contact_max) break;
        if (M.export_rank) o = M.export_rank[o];  // the buffer was reordered by nb2_contacts_sort
#pragma unroll
        for (int k = 0; k < 6; ++k) out.force[6 * size_t(o) + k] = M.contact_impulse[k * T + slot0 + c] * inv_dt;
    }
}

// Stand-alone integrate_bodies (reference SolverBase.integrate_bodies, solver.py:267-307): one thread per body.
__global__ void __launch_bounds__(256) integrate_bodies_kernel(nb2_model_desc d, nb2_state_view sin, nb2_state_view sout,
                                                                float angular_damping, float dt) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= d.body_count) return;
    Xf X = ldx(sin.body_q + 7 * b);
    V3 v0 = ld3(sin.body_qd + 6 * b), w0 = ld3(sin.body_qd + 6 * b + 3);
    if ((d.body_flags[b] & BODY_KINEMATIC) != 0) {
        stx(sout.body_q + 7 * b, X);
        st3(sout.body_qd + 6 * b, v0);
        st3(sout.body_qd + 6 * b + 3, w0);
        return;
    }
    V3 f0 = ld3(sin.body_f + 6 * b), t0 = ld3(sin.body_f + 6 * b + 3);
    const V3 com = ld3(d.body_com + 3 * b);
    const float inv_mass = d.body_inv_mass[b];
    const M33 inertia = ldm(d.body_inertia + 9 * b), inv_inertia = ldm(d.body_inv_inertia + 9 * b);
    int wi = d.body_world[b];
    if (wi < 0) wi += d.gravity_count;
    const V3 g = ld3(d.gravity + 3 * wi);
    const V3 x_com = X.p + qrot(X.q, com);
    const V3 v1 = v0 + (f0 * inv_mass + g * (inv_mass != 0.0f ? 1.0f : 0.0f)) * dt;
    const V3 x1 = x_com + v1 * dt;
    const V3 wb = qrot_inv(X.q, w0);
    const V3 tb = qrot_inv(X.q, t0) - cross(wb, mv(inertia, wb));
    V3 w1 = qrot(X.q, wb + mv(inv_inertia, tb) * dt);
    const Q4 r1 = qunit(qadd(X.q, qscale(qscale(qmul(Q4(w1.x, w1.y, w1.z, 0.0f), X.q), 0.5f), dt)));
    w1 *= 1.0f - angular_damping * dt;
    stx(sout.body_q + 7 * b, Xf(x1 - qrot(r1, com), r1));
    st3(sout.body_qd + 6 * b, v1);
    st3(sout.body_qd + 6 * b + 3, w1);
}

template <int L, bool EX, int WARPS>
static nb2_status launch_xpbd_W(nb2_model* m, const nb2_xpbd_params& p, const nb2_state_view& in, const nb2_state_view& out,
                                const nb2_control_view& ctl, int use_contacts, float dt, cudaStream_t s) {
    const DevModel& M = m->dev;
    constexpr int NE = (32 / L) * WARPS;
    const int blocks = (M.env_count + NE - 1) / NE;
    // contact records per env: the tightest bound the host knows (sum of the pairs' own maxima after nb2_collide; the
    // whole slot range after nb2_contacts_import, whose buffers may hold anything)
    const int contact_cap = m->contacts_imported ? M.max_env_contact_slots : std::min(M.max_env_contact_slots, m->max_env_contacts);
    if (M.max_env_bodies > 32000) {
        set_error("xpbd_step: environment too large for the fused shared-memory kernel (bodies per env)");
        return NB2_ERR_CAPACITY;
    }
    // Budget: the CTAs of one SM share 227 KB (+1 KB reserved each); the batch wants >= ceil(envs / (G * 148)) resident warps per SM to
    // stay a single wave.  The per-joint cache rides along when it does not cost that residency.
    bool joint_cache = false;
    XpbdPlan plan = xpbd_plan(NE, M.max_env_bodies, M.max_env_joints, contact_cap, EX, false);
    if (M.d.joint_count > 0) {
        const XpbdPlan with_cache = xpbd_plan(NE, M.max_env_bodies, M.max_env_joints, contact_cap, EX, true);
        const int want_ctas = (14 + WARPS - 1) / WARPS;  // 14 warps per SM keep 4096 two-env warps in one wave
        if ((size_t(with_cache.total) * sizeof(float) + 1024) * want_ctas <= 227 * 1024 || size_t(plan.total) * sizeof(float) * want_ctas > 227 * 1024) {
            if (size_t(with_cache.total) * sizeof(float) <= 220 * 1024) {
                plan = with_cache;
                joint_cache = true;
            }
        }
    }
    // contact-constant cache: as many contacts per env as still fit (up to the contact bound), keeping the residency above
    int contact_cache = 0;
    {
        const int want_ctas = (14 + WARPS - 1) / WARPS;
        const size_t budget = (size_t(227) * 1024) / want_ctas - 1024 - 64;
        const size_t base = size_t(plan.total) * sizeof(float);
        if (use_contacts && base < budget) {
            contact_cache = int(std::min<size_t>((budget - base) / (size_t(NE) * CC_SIZE * sizeof(float)), size_t(contact_cap)));
            if (contact_cache > 0)
                plan = xpbd_plan(NE, M.max_env_bodies, M.max_env_joints, contact_cap, EX, joint_cache, contact_cache);
        }
    }
    const size_t smem = size_t(plan.total) * sizeof(float);
    if (smem > 220 * 1024 + 6 * 1024) {
        set_error("xpbd_step: environment too large for the fused shared-memory kernel (bodies/contacts per env)");
        return NB2_ERR_CAPACITY;
    }
    if (smem > 48 * 1024)
        NB2_CUDA_CHECK(cudaFuncSetAttribute(xpbd_step_kernel<L, EX, WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    // ask for the largest shared-memory carve-out so that ~14-16 warps' worth of CTAs fit per SM
    NB2_CUDA_CHECK(cudaFuncSetAttribute(xpbd_step_kernel<L, EX, WARPS>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    xpbd_step_kernel<L, EX, WARPS><<<blocks, 32 * WARPS, smem, s>>>(M, p, in, out, ctl, use_contacts, dt, joint_cache, contact_cap, contact_cache);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

// Warps per CTA.  Measured on B200 (profiles/r2b_xpbd_ab.txt, 4096 quadruped envs): 1 / 2 / 4 warps 166 us, 7 warps 160 us,
// 14 warps 155 us, and 148 us with the per-iteration CTA barrier - the more warps walk the same code together, the fewer times the
// instruction stream is fetched.  The launch takes the largest compiled width that the batch can fill on every SM
// (14 = one CTA per SM for 4096 two-env warps) and falls back when shared memory does not allow it.
template <int L, bool EX>
static nb2_status launch_xpbd_L(nb2_model* m, const nb2_xpbd_params& p, const nb2_state_view& in, const nb2_state_view& out,
                                const nb2_control_view& ctl, int use_contacts, float dt, cudaStream_t s) {
    const long long per_sm = warps_per_sm(m, L);
    int warps = per_sm <= 1 ? 1 : (per_sm <= 4 ? 4 : 14);
    // shared-memory fit (the per-CTA plan grows with the warp count)
    auto fits = [&](int w) {
        const int ne = (32 / L) * w;
        const int cap = m->contacts_imported ? m->dev.max_env_contact_slots : std::min(m->dev.max_env_contact_slots, m->max_env_contacts);
        return size_t(xpbd_plan(ne, m->dev.max_env_bodies, m->dev.max_env_joints, cap, EX, false).total) * sizeof(float) <= 200 * 1024;
    };
    if (warps >= 14 && !fits(14)) warps = 4;
    if (warps >= 4 && warps < 14 && !fits(4)) warps = 1;
    if (warps >= 14) return launch_xpbd_W<L, EX, 14>(m, p, in, out, ctl, use_contacts, dt, s);
    if (warps >= 4) return launch_xpbd_W<L, EX, 4>(m, p, in, out, ctl, use_contacts, dt, s);
    return launch_xpbd_W<L, EX, 1>(m, p, in, out, ctl, use_contacts, dt, s);
}

nb2_status launch_xpbd_step(nb2_model* m, const nb2_xpbd_params& p, const nb2_state_view& in, const nb2_state_view& out,
                            const nb2_control_view& ctl, int use_contacts, float dt, cudaStream_t s) {
    const DevModel& M = m->dev;
    if (M.d.body_count == 0) return NB2_OK;
    if (!in.body_q || !in.body_qd || !in.body_f || !out.body_q || !out.body_qd) {
        set_error("nb2_xpbd_step: state arrays are NULL");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (M.d.joint_count > 0 && (!ctl.joint_f || !ctl.joint_target_q || !ctl.joint_target_qd)) {
        set_error("nb2_xpbd_step: control arrays are NULL");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (p.enable_restitution && !M.d.shape_material_restitution) {
        set_error("nb2_xpbd_step: enable_restitution needs model.shape_material_restitution");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    const bool ex = p.enable_restitution || p.compute_body_velocity_from_position_delta || out.body_parent_f != nullptr ||
                    ((use_contacts & NB2_XPBD_CONTACT_IMPULSE) && (use_contacts & NB2_XPBD_USE_CONTACTS));
#define XPBD_DISPATCH(LANES)                                                                        \
    return ex ? launch_xpbd_L<LANES, true>(m, p, in, out, ctl, use_contacts, dt, s)                     \
              : launch_xpbd_L<LANES, false>(m, p, in, out, ctl, use_contacts, dt, s)
    switch (m->lanes_per_env) {
        case 8: XPBD_DISPATCH(8);
        case 16: XPBD_DISPATCH(16);
        default: XPBD_DISPATCH(32);
    }
#undef XPBD_DISPATCH
}

nb2_status launch_xpbd_update_contacts(nb2_model* m, const nb2_contacts_view& contacts, cudaStream_t s) {
    const DevModel& M = m->dev;
    NB2_CUDA_CHECK(cudaMemsetAsync(contacts.force, 0, size_t(contacts.rigid_contact_max) * 6 * sizeof(float), s));
    if (M.env_count == 0) return NB2_OK;
    xpbd_update_contacts_kernel<<<(M.env_count + 3) / 4, 128, 0, s>>>(M, contacts, 1.0f / m->xpbd_impulse_dt);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

nb2_status launch_integrate_bodies(nb2_model* m, const nb2_state_view& in, const nb2_state_view& out, float angular_damping, float dt,
                                   cudaStream_t s) {
    const nb2_model_desc& d = m->dev.d;
    if (d.body_count == 0) return NB2_OK;
    integrate_bodies_kernel<<<(d.body_count + 255) / 256, 256, 0, s>>>(d, in, out, angular_damping, dt);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

}  // namespace nb2
