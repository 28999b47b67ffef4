// nb2_featherstone.cu - fused articulated-body step for sm_100a (reference SolverFeatherstone.step,
// solvers/featherstone/solver_featherstone.py:461-1066; kernels in solvers/featherstone/kernels.py).
//
// The reference spends ~16 launches per substep, walks every articulation with ONE thread (FK, RNEA forward /
// backward), materialises a dense 6nj x 6nj mass matrix M (97 % zeros) plus J and P = M J in HBM and multiplies
// them with one thread per articulation (kernels.py:1504-1538: 78x78x18 serial MACs).  Here one launch does the
// whole step; a sub-warp group of L lanes owns one environment and keeps every intermediate in shared memory:
//
//   eval_rigid_fk                  :687-728     joint lanes, level by level (joints of equal tree depth in parallel)
//   public->internal qd / joint_f  :924-975, :1069-1088, :893-921
//   eval_rigid_id (RNEA forward)   :1241-1317   level-parallel; spatial inertia T^T I T by blocks (T = [[R,S],[0,R]])
//   eval_body_contact (penalty)    semi_implicit/kernels_contact.py:381-556   body lanes, ordered by contact index
//   eval_rigid_tau (RNEA backward) :1320-1418   level-parallel, children folded into the parent in descending joint order
//   H = J^T M J                    :1422-1501, :1655-1687   never forms M, J or P: H[a][b] = sum over the joints i below
//                                  both dofs of S_a . (I_s[i] S_b), accumulated in the reference's k-order
//   dense_cholesky / dense_subs    :1690-1781   column-parallel factorisation, serial substitutions (order-preserving)
//   integrate_generalized_joints   :1849-1893 (jcalc_integrate :464-630)
//   eval_fk_with_velocity_conversion :1987-2149, internal->public qd :1015-1066
//
// Every sum is taken in the order of the reference's serial loops (structural zeros skipped, which is exact), so the
// strict-fp build reproduces the CPU oracle bit for bit.  Tensor cores (north_star: "only for the small dense
// mass-matrix factor/solve") would need TF32 or 3xTF32 splits and cannot meet bit-parity; with H at 18x18 the stage is
// ~9 k MACs per env, latency- not throughput-bound, so it stays on the FP32 pipe (DESIGN.md §3).

#include "nb2_internal.cuh"
#include "nb2_math.cuh"

namespace nb2 {

enum { FJ_PRISMATIC = 0, FJ_REVOLUTE = 1, FJ_BALL = 2, FJ_FIXED = 3, FJ_FREE = 4, FJ_DISTANCE = 5, FJ_D6 = 6 };

struct S6 {
    float v[6];
    NB2_DEV S6() {
#pragma unroll
        for (int i = 0; i < 6; ++i) v[i] = 0.f;
    }
    NB2_DEV S6(V3 a, V3 b) { v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = b.x; v[4] = b.y; v[5] = b.z; }
    NB2_DEV V3 top() const { return V3(v[0], v[1], v[2]); }
    NB2_DEV V3 bot() const { return V3(v[3], v[4], v[5]); }
};
NB2_DEV S6 ld6(const float* p) {
    S6 s;
#pragma unroll
    for (int i = 0; i < 6; ++i) s.v[i] = p[i];
    return s;
}
NB2_DEV void st6(float* p, const S6& s) {
#pragma unroll
    for (int i = 0; i < 6; ++i) p[i] = s.v[i];
}
NB2_DEV S6 operator+(const S6& a, const S6& b) {
    S6 r;
#pragma unroll
    for (int i = 0; i < 6; ++i) r.v[i] = a.v[i] + b.v[i];
    return r;
}
NB2_DEV S6 operator-(const S6& a, const S6& b) {
    S6 r;
#pragma unroll
    for (int i = 0; i < 6; ++i) r.v[i] = a.v[i] - b.v[i];
    return r;
}
NB2_DEV S6 operator*(const S6& a, float s) {
    S6 r;
#pragma unroll
    for (int i = 0; i < 6; ++i) r.v[i] = a.v[i] * s;
    return r;
}
NB2_DEV float dot6(const S6& a, const S6& b) {
    return a.v[0] * b.v[0] + a.v[1] * b.v[1] + a.v[2] * b.v[2] + a.v[3] * b.v[3] + a.v[4] * b.v[4] + a.v[5] * b.v[5];
}
NB2_DEV S6 twist_xf(const Xf& t, const S6& x) {  // math/spatial.py:82-105
    V3 w = qrot(t.q, x.bot());
    V3 v = qrot(t.q, x.top()) + cross(t.p, w);
    return S6(v, w);
}
NB2_DEV S6 scross(const S6& a, const S6& b) {
    V3 w = cross(a.bot(), b.bot());
    V3 v = cross(a.bot(), b.top()) + cross(a.top(), b.bot());
    return S6(v, w);
}
NB2_DEV S6 scross_dual(const S6& a, const S6& b) {
    V3 w = cross(a.bot(), b.bot()) + cross(a.top(), b.top());
    V3 v = cross(a.bot(), b.top());
    return S6(v, w);
}
NB2_DEV S6 m66v(const float* I, const S6& b) {  // dense 6x6 (row-major in shared memory) times vector, column order
    S6 r;
#pragma unroll
    for (int i = 0; i < 6; ++i) r.v[i] = I[6 * i] * b.v[0];
#pragma unroll
    for (int c = 1; c < 6; ++c)
#pragma unroll
        for (int i = 0; i < 6; ++i) r.v[i] += I[6 * i + c] * b.v[c];
    return r;
}
NB2_DEV Q4 q_axis_angle(V3 axis, float angle) {
    float half = angle * 0.5f;
    float w = cos_w(half), s = sin_w(half);
    V3 v = axis * s;
    return Q4(v.x, v.y, v.z, w);
}

// transform_spatial_inertia (kernels.py:66-138) for I = blockdiag(m 1, Ic): T^T I T with T = [[R, S], [0, R]],
// R / S from the inverse transform.  Sums follow the dense k-order of the reference with structural zeros dropped.
NB2_DEV void spatial_inertia(const Xf& t, float mass, const M33& Ic, float* out) {
    const Xf ti = xinv(t);
    const M33 R = qmat(ti.q);
    const V3 p = ti.p;
    M33 S;  // skew(p) @ R
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        S.a[0 + j] = (-p.z) * R.a[3 + j] + p.y * R.a[6 + j];
        S.a[3 + j] = p.z * R.a[0 + j] + (-p.x) * R.a[6 + j];
        S.a[6 + j] = (-p.y) * R.a[0 + j] + p.x * R.a[3 + j];
    }
    float A[6][6];  // A = T^T I
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            A[i][j] = R.a[3 * j + i] * mass;
            A[i][j + 3] = 0.0f;
            A[i + 3][j] = S.a[3 * j + i] * mass;
            float s = R.a[0 + i] * Ic.a[0 + j];
            s += R.a[3 + i] * Ic.a[3 + j];
            s += R.a[6 + i] * Ic.a[6 + j];
            A[i + 3][j + 3] = s;
        }
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            float s = A[i][0] * R.a[0 + j];
            s += A[i][1] * R.a[3 + j];
            s += A[i][2] * R.a[6 + j];
            out[6 * i + j] = s;
            float u = A[i][0] * S.a[0 + j];
            u += A[i][1] * S.a[3 + j];
            u += A[i][2] * S.a[6 + j];
            if (i >= 3) {
                u += A[i][3] * R.a[0 + j];
                u += A[i][4] * R.a[3 + j];
                u += A[i][5] * R.a[6 + j];
            }
            out[6 * i + j + 3] = u;
        }
}

NB2_DEV float joint_force(float q, float qd, float tq, float tqd, float ke, float kd, float lo, float up, float lke, float lkd, float damping) {
    float limit_f = 0.0f, damping_f = 0.0f;
    float target_f = ke * (tq - q) + kd * (tqd - qd);
    if (q < lo) {
        limit_f = lke * (lo - q);
        damping_f = -lkd * qd;
        target_f = 0.0f;
    } else if (q > up) {
        limit_f = lke * (up - q);
        damping_f = -lkd * qd;
        target_f = 0.0f;
    }
    float passive_f = -damping * qd;
    return limit_f + damping_f + target_f + passive_f;
}

// wp.quat_from_matrix of the matrix whose COLUMNS are c0, c1, c2 (trace branch, else the largest diagonal element; normalized)
NB2_DEV Q4 q_from_cols(V3 c0, V3 c1, V3 c2) {
    const float m00 = c0.x, m10 = c0.y, m20 = c0.z, m01 = c1.x, m11 = c1.y, m21 = c1.z, m02 = c2.x, m12 = c2.y, m22 = c2.z;
    const float tr = m00 + m11 + m22;
    float x, y, z, w, h;
    if (tr >= 0.0f) {
        h = sqrtf(tr + 1.0f);
        w = 0.5f * h;
        h = 0.5f / h;
        x = (m21 - m12) * h;
        y = (m02 - m20) * h;
        z = (m10 - m01) * h;
    } else {
        int md = 0;
        if (m11 > m00) md = 1;
        if (m22 > (md == 0 ? m00 : m11)) md = 2;
        if (md == 0) {
            h = sqrtf((m00 - (m11 + m22)) + 1.0f);
            x = 0.5f * h;
            h = 0.5f / h;
            y = (m01 + m10) * h;
            z = (m20 + m02) * h;
            w = (m21 - m12) * h;
        } else if (md == 1) {
            h = sqrtf((m11 - (m22 + m00)) + 1.0f);
            y = 0.5f * h;
            h = 0.5f / h;
            z = (m12 + m21) * h;
            x = (m01 + m10) * h;
            w = (m02 - m20) * h;
        } else {
            h = sqrtf((m22 - (m00 + m11)) + 1.0f);
            z = 0.5f * h;
            h = 0.5f / h;
            x = (m20 + m02) * h;
            y = (m12 + m21) * h;
            w = (m10 - m01) * h;
        }
    }
    return qunit(Q4(x, y, z, w));
}
// transform_2d_rotational_axes (sim/articulation.py:37-58): D6 joints with exactly two angular axes
NB2_DEV void axes2(V3 a0, V3 a1, float q0, V3& o0, V3& o1) {
    const Q4 q_off = q_from_cols(a0, a1, cross(a0, a1));
    const V3 l0 = qrot(q_off, V3(1.f, 0.f, 0.f)), l1 = qrot(q_off, V3(0.f, 1.f, 0.f));
    o0 = l0;
    o1 = qrot(q_axis_angle(l0, q0), l1);
}
NB2_DEV void axes3(V3 a0, V3 a1, V3 a2, float q0, float q1, V3& o0, V3& o1, V3& o2) {  // transform_3d_rotational_axes
    Q4 q_0 = q_axis_angle(a0, q0);
    V3 a1w = qrot(q_0, a1);
    Q4 q_1 = q_axis_angle(a1w, q1);
    V3 a2w = qrot(qmul(q_1, q_0), a2);
    o0 = a0; o1 = a1w; o2 = a2w;
}

// jcalc_transform (kernels.py:142-238)
NB2_DEV Xf joint_transform(const nb2_model_desc& d, int type, int axis_start, int lin, int ang, const float* jq, int qs) {
    if (type == FJ_PRISMATIC) return Xf(ld3(d.joint_axis + 3 * axis_start) * jq[qs], Q4());
    if (type == FJ_REVOLUTE) return Xf(V3(), q_axis_angle(ld3(d.joint_axis + 3 * axis_start), jq[qs]));
    if (type == FJ_BALL) return Xf(V3(), Q4(jq[qs], jq[qs + 1], jq[qs + 2], jq[qs + 3]));
    if (type == FJ_FREE || type == FJ_DISTANCE) return Xf(V3(jq[qs], jq[qs + 1], jq[qs + 2]), Q4(jq[qs + 3], jq[qs + 4], jq[qs + 5], jq[qs + 6]));
    if (type == FJ_D6) {
        V3 pos;
        Q4 rot;
        for (int k = 0; k < 3; ++k)
            if (lin > k) pos += ld3(d.joint_axis + 3 * (axis_start + k)) * jq[qs + k];
        const int ia = axis_start + lin, iq = qs + lin;
        if (ang == 1) rot = q_axis_angle(ld3(d.joint_axis + 3 * ia), jq[iq]);
        if (ang == 2) {  // compute_2d_rotational_dofs (sim/articulation.py:61-82)
            V3 w0, w1;
            axes2(ld3(d.joint_axis + 3 * ia), ld3(d.joint_axis + 3 * (ia + 1)), jq[iq], w0, w1);
            rot = qmul(q_axis_angle(w1, jq[iq + 1]), q_axis_angle(w0, jq[iq]));
        }
        if (ang == 3) {
            V3 w0, w1, w2;
            axes3(ld3(d.joint_axis + 3 * ia), ld3(d.joint_axis + 3 * (ia + 1)), ld3(d.joint_axis + 3 * (ia + 2)), jq[iq], jq[iq + 1], w0, w1, w2);
            rot = qmul(qmul(q_axis_angle(w2, jq[iq + 2]), q_axis_angle(w1, jq[iq + 1])), q_axis_angle(w0, jq[iq]));
        }
        return Xf(pos, rot);
    }
    return Xf();
}

struct FsSmem {
    float *bq, *bqc, *vs, *as, *fb, *ft, *fe, *qdfk, *Is, *so, *fs, *S, *qd_in, *jf, *tau, *qdd, *qd_out, *H, *jq, *P;
    // joint headers staged once per substep: the level passes index these instead of going to global memory for every joint's
    // type / parent / child / depth / offsets in every pass (25 % of the stall samples were those L1 round trips)
    int *h_type, *h_parent, *h_child, *h_depth, *h_dim, *h_q, *h_qd;
};
NB2_DEV size_t fs_smem_floats(const DevModel& M) {
    const size_t n = size_t(M.max_env_bodies) * (7 + 7 + 6 * 6 + 36 + 3 + 6) + size_t(M.max_env_joints) * 6 +
                     size_t(M.max_env_dofs) * (6 + 5) + size_t(M.max_env_H) + size_t(M.max_env_coords) + size_t(M.max_env_joints) * 8 + 2;
    return (n + 1) & ~size_t(1);
}
NB2_DEV FsSmem fs_carve(float* base, const DevModel& M) {
    FsSmem s;
    const int nb = M.max_env_bodies, nj = M.max_env_joints, nd = M.max_env_dofs;
    float* p = base;
    s.bq = p; p += nb * 7;
    s.bqc = p; p += nb * 7;
    s.vs = p; p += nb * 6;
    s.as = p; p += nb * 6;
    s.fb = p; p += nb * 6;
    s.ft = p; p += nb * 6;
    s.fe = p; p += nb * 6;
    s.qdfk = p; p += nb * 6;
    s.Is = p; p += nb * 36;
    s.so = p; p += nb * 3;
    s.fs = p; p += nj * 6;
    s.S = p; p += nd * 6;
    s.qd_in = p; p += nd;
    s.jf = p; p += nd;
    s.tau = p; p += nd;
    s.qdd = p; p += nd;
    s.qd_out = p; p += nd;
    s.H = p; p += M.max_env_H;
    s.jq = p; p += M.max_env_coords;
    s.P = p; p += nb * 6;
    int* q = reinterpret_cast<int*>(p);
    s.h_type = q; q += nj;
    s.h_parent = q; q += nj;
    s.h_child = q; q += nj;
    s.h_depth = q; q += nj;
    s.h_dim = q; q += 2 * nj;
    s.h_q = q; q += nj + 1;
    s.h_qd = q; q += nj + 1;
    return s;
}

// ---- tensor-core H = J^T (M J) (reference use_tile_gemm: eval_dense_gemm_tile / the fused tile kernels, featherstone/kernels.py:
// 1568-1652) -------------------------------------------------------------------------------------------------------------------------
// One warp forms the H of ONE articulation at a time with mma.sync.m16n8k8 (TF32 inputs, FP32 accumulate).  The K dimension is
// walked body by body (6 of the 8 k-slots used): per body i
//     P_i [6 x n]  = I_i [6 x 6] . J_i [6 x n]      1 M-tile x 3 N-tiles     (J_i[:, b] = S_b if joint(b) is an ancestor-or-self of i)
//     H  [n x n]  += J_i^T [n x 6] . P_i [6 x n]    2 M-tiles x 3 N-tiles
// with every product taken as the 3xTF32 split  a.b ~ a_lo.b_hi + a_hi.b_lo + a_hi.b_hi  (a_hi = tf32(a), a_lo = tf32(a - a_hi)),
// which carries ~2^-21 relative error per product - H agrees with the FP32 path to ~1e-6, not bit for bit, which is why the path is
// opt-in (SolverFeatherstone(use_tile_gemm=True)).  n <= 24 (3 N-tiles, 2 M-tiles): checked by the launcher.
#define NB2_GPU_FN __device__ __forceinline__
NB2_GPU_FN unsigned to_tf32(float x) {
    unsigned r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return r;
}
NB2_GPU_FN void mma_tf32(float (&c)[4], const unsigned (&a)[4], const unsigned (&b)[2]) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
NB2_GPU_FN void mma_3xtf32(float (&c)[4], const float (&a)[4], const float (&b)[2]) {
    unsigned ah[4], al[4], bh[2], bl[2];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        ah[i] = to_tf32(a[i]);
        al[i] = to_tf32(a[i] - __uint_as_float(ah[i]));
    }
#pragma unroll
    for (int i = 0; i < 2; ++i) {
        bh[i] = to_tf32(b[i]);
        bl[i] = to_tf32(b[i] - __uint_as_float(bh[i]));
    }
    mma_tf32(c, al, bh);  // small terms first
    mma_tf32(c, ah, bl);
    mma_tf32(c, ah, bh);
}
// S: the articulation's motion subspaces (6 floats per dof), Is: its bodies' spatial inertias (36 floats each, body i == joint i),
// anc / dofj: ancestor masks and dof -> joint table (articulation-local), Pbuf: 6 x 24 floats of warp scratch, H: n x n output.
__device__ __noinline__ void tile_mass_matrix(const float* S, const float* Is, const unsigned long long* anc, const signed char* dofj, int anj,
                                              int n, float* Pbuf, float* H) {
    const int lane = threadIdx.x & 31, gq = lane >> 2, tq = lane & 3;
    float acc[2][3][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 3; ++nt)
#pragma unroll
            for (int k = 0; k < 4; ++k) acc[mt][nt][k] = 0.0f;
    for (int i = 0; i < anj; ++i) {
        const unsigned long long am = anc[i];
        const float* I = Is + 36 * i;
        // A = I_i as a 16 x 8 tile: rows gq / gq + 8 (only rows < 6 exist), columns tq / tq + 4
        float a1[4] = {gq < 6 ? I[6 * gq + tq] : 0.0f, 0.0f, (gq < 6 && tq < 2) ? I[6 * gq + tq + 4] : 0.0f, 0.0f};
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
            const int b = 8 * nt + gq;  // this lane's column of J_i
            const bool on = b < n && ((am >> dofj[b < n ? b : 0]) & 1ull);
            float b1[2] = {on ? S[6 * b + tq] : 0.0f, (on && tq < 2) ? S[6 * b + tq + 4] : 0.0f};
            float c[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            mma_3xtf32(c, a1, b1);
            if (gq < 6) {  // C rows gq: P_i[gq][8 nt + 2 tq], [.. + 1]
                Pbuf[gq * 24 + 8 * nt + 2 * tq] = c[0];
                Pbuf[gq * 24 + 8 * nt + 2 * tq + 1] = c[1];
            }
        }
        __syncwarp();
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) {
            const int r0 = 16 * mt + gq, r1 = r0 + 8;  // rows of H = columns of J_i
            const bool on0 = r0 < n && ((am >> dofj[r0 < n ? r0 : 0]) & 1ull), on1 = r1 < n && ((am >> dofj[r1 < n ? r1 : 0]) & 1ull);
            float a2[4] = {on0 ? S[6 * r0 + tq] : 0.0f, on1 ? S[6 * r1 + tq] : 0.0f, (on0 && tq < 2) ? S[6 * r0 + tq + 4] : 0.0f,
                           (on1 && tq < 2) ? S[6 * r1 + tq + 4] : 0.0f};
#pragma unroll
            for (int nt = 0; nt < 3; ++nt) {
                float b2[2] = {Pbuf[tq * 24 + 8 * nt + gq], tq < 2 ? Pbuf[(tq + 4) * 24 + 8 * nt + gq] : 0.0f};
                mma_3xtf32(acc[mt][nt], a2, b2);
            }
        }
        __syncwarp();
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
        for (int nt = 0; nt < 3; ++nt) {
            const int r0 = 16 * mt + gq, r1 = r0 + 8, c0 = 8 * nt + 2 * tq;
            if (r0 < n && c0 < n) H[r0 * n + c0] = acc[mt][nt][0];
            if (r0 < n && c0 + 1 < n) H[r0 * n + c0 + 1] = acc[mt][nt][1];
            if (r1 < n && c0 < n) H[r1 * n + c0] = acc[mt][nt][2];
            if (r1 < n && c0 + 1 < n) H[r1 * n + c0 + 1] = acc[mt][nt][3];
        }
    __syncwarp();
}

// PF: also write State.body_parent_f (compute_body_parent_f, featherstone/kernels.py:2371-2416) - a second instantiation, so
// that the plain step's code is untouched (the same arrangement as xpbd_step_kernel<L, EX>).
//
// WARPS warps per CTA, each warp = 32/L environments, with CTA barriers at the phase boundaries (NB2_PHASE): not needed for
// correctness - a sub-warp group owns its environment - they keep the CTA's warps on the same stretch of this ~9 000-instruction
// kernel, so the instruction stream is fetched once per CTA instead of once per warp (measured on xpbd_step_kernel:
// profiles/r2b_xpbd_ab.txt).
#define NB2_PHASE()                       \
    do {                                  \
        if (WARPS > 1) __syncthreads();   \
    } while (0)
template <int L, bool PF, int WARPS, bool TILE>
__global__ void __launch_bounds__(32 * WARPS, (WARPS >= 14 ? 1 : 14 / WARPS))
featherstone_step_kernel(DevModel M, nb2_featherstone_params P, nb2_state_view sin, nb2_state_view sout, nb2_control_view ctl, int use_contacts,
                         int update_mass, float dt) {
    constexpr int G = 32 / L;
    extern __shared__ float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int grp = lane / L, l = lane % L;
    const int env = (blockIdx.x * WARPS + warp) * G + grp;
    const bool live = env < M.env_count;
    // groups run different trip counts (articulations / dofs per env), so barriers cover one group only
    const unsigned gmask = (L == 32) ? 0xffffffffu : (((1u << L) - 1u) << (grp * L));
    const nb2_model_desc& d = M.d;
    const FsSmem sm = fs_carve(smem + size_t(warp * G + grp) * fs_smem_floats(M), M);

    int b0 = 0, nb = 0, j0 = 0, nj = 0, a0 = 0, na = 0, d0 = 0, nd = 0, c0 = 0, ncoord = 0, slot0 = 0, nc = 0;
    if (live) {
        b0 = M.env_body_start[env];
        nb = M.env_body_start[env + 1] - b0;
        j0 = M.env_joint_start[env];
        nj = M.env_joint_start[env + 1] - j0;
        a0 = M.env_art_start[env];
        na = M.env_art_start[env + 1] - a0;
        d0 = d.joint_qd_start[j0];
        nd = d.joint_qd_start[j0 + nj] - d0;
        c0 = d.joint_q_start[j0];
        ncoord = d.joint_q_start[j0 + nj] - c0;
        slot0 = M.env_slot_start[env];
        nc = use_contacts ? M.env_contact_count[env] : 0;
    }
    const size_t T = size_t(M.slot_total);
    const float* cb = M.cb;
    for (int j = l; j < nj; j += L) {
        const int gj = j0 + j;
        sm.h_type[j] = d.joint_type[gj];
        sm.h_parent[j] = d.joint_parent[gj];
        sm.h_child[j] = d.joint_child[gj];
        sm.h_depth[j] = M.joint_depth[gj];
        sm.h_dim[2 * j] = d.joint_dof_dim[2 * gj];
        sm.h_dim[2 * j + 1] = d.joint_dof_dim[2 * gj + 1];
        sm.h_q[j] = d.joint_q_start[gj];
        sm.h_qd[j] = d.joint_qd_start[gj];
    }
    if (l == 0 && live) {
        sm.h_q[nj] = d.joint_q_start[j0 + nj];
        sm.h_qd[nj] = d.joint_qd_start[j0 + nj];
    }
    // views indexed by GLOBAL joint id, like the model arrays they shadow
    const int *jtype = sm.h_type - j0, *jparent = sm.h_parent - j0, *jchild = sm.h_child - j0, *jdepth = sm.h_depth - j0,
              *jdim = sm.h_dim - 2 * j0, *jqs = sm.h_q - j0, *jqds = sm.h_qd - j0;
    __syncwarp(gmask);

    // ---- body_f_ext = body_f; zero scratch ------------------------------------------------------
    for (int b = l; b < nb; b += L) {
#pragma unroll
        for (int k = 0; k < 6; ++k) {
            sm.fe[6 * b + k] = sin.body_f[6 * (b0 + b) + k];
            sm.ft[6 * b + k] = 0.f;
            sm.fb[6 * b + k] = 0.f;
        }
    }
    __syncwarp(gmask);
    // ---- per joint: public -> internal joint_f, FREE/DISTANCE wrench into body_f_ext -------------
    for (int j = l; j < nj; j += L) {
        const int gj = j0 + j, type = jtype[gj];
        const int qd0 = jqds[gj], qd1 = jqds[gj + 1];
        if (type == FJ_FREE || type == FJ_DISTANCE) {
            const int child = jchild[gj] - b0;
#pragma unroll
            for (int k = 0; k < 6; ++k) sm.fe[6 * child + k] += ctl.joint_f[qd0 + k];  // one inbound joint per body
            for (int i = qd0; i < qd1; ++i) sm.jf[i - d0] = 0.0f;
        } else {
            for (int i = qd0; i < qd1; ++i) sm.jf[i - d0] = ctl.joint_f[i];
        }
    }
    // ---- eval_rigid_fk: joint-local transforms for all joints at once, then the tree recurrence level by level ----------------
    // (scratch: X_j(q) and X_cj^-1 live in the spatial-inertia block of the joint's body, which is unused until the RNEA pass)
    for (int j = l; j < nj; j += L) {
        const int gj = j0 + j;
        const Xf X_j = joint_transform(d, jtype[gj], jqds[gj], jdim[2 * gj], jdim[2 * gj + 1],
                                       sin.joint_q, jqs[gj]);
        stx(sm.Is + 36 * j, X_j);
        stx(sm.Is + 36 * j + 7, xinv(ldx(d.joint_X_c + 7 * gj)));
    }
    __syncwarp(gmask);
    for (int lvl = 0; lvl <= M.max_depth; ++lvl) {
        for (int j = l; j < nj; j += L) {
            const int gj = j0 + j;
            if (jdepth[gj] != lvl) continue;
            const int parent = jparent[gj], child = jchild[gj] - b0;
            Xf X_wpj = ldx(d.joint_X_p + 7 * gj);
            if (parent >= 0) X_wpj = xmul(ldx(sm.bq + 7 * (parent - b0)), X_wpj);
            const Xf X_wc = xmul(xmul(X_wpj, ldx(sm.Is + 36 * j)), ldx(sm.Is + 36 * j + 7));
            const Xf X_sm = xmul(X_wc, Xf(ld3(d.body_com + 3 * (b0 + child)), Q4()));
            stx(sm.bq + 7 * child, X_wc);
            stx(sm.bqc + 7 * child, X_sm);
            stx(sin.body_q + 7 * (b0 + child), X_wc);  // the reference refreshes state_in.body_q (solver_featherstone.py:511)
        }
        __syncwarp(gmask);
    }
    // ---- public -> internal joint_qd ------------------------------------------------------------------
    for (int j = l; j < nj; j += L) {
        const int gj = j0 + j, type = jtype[gj];
        const int qd0 = jqds[gj], qd1 = jqds[gj + 1];
        if (type != FJ_FREE && type != FJ_DISTANCE) {
            for (int i = qd0; i < qd1; ++i) sm.qd_in[i - d0] = sin.joint_qd[i];
            continue;
        }
        const int parent = jparent[gj], child = jchild[gj] - b0;
        Xf X_wpj = ldx(d.joint_X_p + 7 * gj);
        if (parent >= 0) X_wpj = xmul(ldx(sm.bq + 7 * (parent - b0)), X_wpj);
        const V3 x_com = xpoint(ldx(sm.bq + 7 * child), ld3(d.body_com + 3 * (b0 + child)));
        const V3 r = qrot_inv(X_wpj.q, x_com - X_wpj.p);
        const V3 v_com(sin.joint_qd[qd0], sin.joint_qd[qd0 + 1], sin.joint_qd[qd0 + 2]);
        const V3 omega(sin.joint_qd[qd0 + 3], sin.joint_qd[qd0 + 4], sin.joint_qd[qd0 + 5]);
        const V3 v_int = v_com - cross(omega, r);
        float* o = sm.qd_in + (qd0 - d0);
        o[0] = v_int.x; o[1] = v_int.y; o[2] = v_int.z; o[3] = omega.x; o[4] = omega.y; o[5] = omega.z;
    }
    __syncwarp(gmask);
    NB2_PHASE();
    // ---- eval_rigid_id (RNEA forward).  Only v_s / a_s recur down the tree; everything else - motion subspaces S, joint
    // velocities v_j, bias terms, spatial inertias - needs the FK poses alone and runs for all joints at once. ---------------
    for (int j = l; j < nj; j += L) {  // A: per-joint quantities (v_j parked in vs[child], c_app in as[child])
        const int gj = j0 + j;
        const int type = jtype[gj], parent = jparent[gj], child = jchild[gj] - b0;
        const int art = d.joint_articulation[gj];
        const int root = d.articulation_start[art];
        V3 solve_origin;
        {
            const int rt = jtype[root];
            if (rt == FJ_FREE || rt == FJ_DISTANCE) solve_origin = ld3(sm.bqc + 7 * (jchild[root] - b0));
        }
        Xf X_wpj = ldx(d.joint_X_p + 7 * gj);
        if (parent >= 0) X_wpj = xmul(ldx(sm.bq + 7 * (parent - b0)), X_wpj);
        const Xf X_s(X_wpj.p - solve_origin, X_wpj.q);
        const int qs = jqs[gj], qds = jqds[gj];
        const int lin = jdim[2 * gj], ang = jdim[2 * gj + 1];
        const float* jqd = sm.qd_in - d0;  // indexed with global dof ids
        float* Sout = sm.S - 6 * d0;
        S6 v_j, c_app;
        if (type == FJ_PRISMATIC) {
            S6 S = twist_xf(X_s, S6(ld3(d.joint_axis + 3 * qds), V3()));
            v_j = S * jqd[qds];
            st6(Sout + 6 * qds, S);
        } else if (type == FJ_REVOLUTE) {
            S6 S = twist_xf(X_s, S6(V3(), ld3(d.joint_axis + 3 * qds)));
            v_j = S * jqd[qds];
            st6(Sout + 6 * qds, S);
        } else if (type == FJ_D6) {
            V3 c_ang;
            for (int k = 0; k < 3; ++k)
                if (lin > k) {
                    S6 S = twist_xf(X_s, S6(ld3(d.joint_axis + 3 * (qds + k)), V3()));
                    v_j = v_j + S * jqd[qds + k];
                    st6(Sout + 6 * (qds + k), S);
                }
            const int iqd = qds + lin, iq = qs + lin;
            if (ang == 1) {
                S6 S = twist_xf(X_s, S6(V3(), ld3(d.joint_axis + 3 * iqd)));
                v_j = v_j + S * jqd[iqd];
                st6(Sout + 6 * iqd, S);
            }
            if (ang == 2) {  // kernels.py:301-311
                V3 w0, w1;
                axes2(ld3(d.joint_axis + 3 * iqd), ld3(d.joint_axis + 3 * (iqd + 1)), sin.joint_q[iq], w0, w1);
                S6 S0 = twist_xf(X_s, S6(V3(), w0)), S1 = twist_xf(X_s, S6(V3(), w1));
                const float q0 = jqd[iqd], q1 = jqd[iqd + 1];
                v_j = v_j + (S0 * q0 + S1 * q1);
                st6(Sout + 6 * iqd, S0);
                st6(Sout + 6 * (iqd + 1), S1);
                c_ang += cross(w0, w1) * (q0 * q1);
            }
            if (ang == 3) {
                V3 w0, w1, w2;
                axes3(ld3(d.joint_axis + 3 * iqd), ld3(d.joint_axis + 3 * (iqd + 1)), ld3(d.joint_axis + 3 * (iqd + 2)), sin.joint_q[iq],
                      sin.joint_q[iq + 1], w0, w1, w2);
                S6 S0 = twist_xf(X_s, S6(V3(), w0)), S1 = twist_xf(X_s, S6(V3(), w1)), S2 = twist_xf(X_s, S6(V3(), w2));
                const float q0 = jqd[iqd], q1 = jqd[iqd + 1], q2 = jqd[iqd + 2];
                v_j = v_j + (S0 * q0 + S1 * q1 + S2 * q2);
                st6(Sout + 6 * iqd, S0);
                st6(Sout + 6 * (iqd + 1), S1);
                st6(Sout + 6 * (iqd + 2), S2);
                c_ang += cross(w0, w1) * (q0 * q1);
                c_ang += cross(w0, w2) * (q0 * q2);
                c_ang += cross(w1, w2) * (q1 * q2);
            }
            c_app = twist_xf(X_s, S6(V3(), c_ang));
        } else if (type == FJ_BALL) {
            S6 S0 = twist_xf(X_s, S6(V3(), V3(1.f, 0.f, 0.f))), S1 = twist_xf(X_s, S6(V3(), V3(0.f, 1.f, 0.f))),
               S2 = twist_xf(X_s, S6(V3(), V3(0.f, 0.f, 1.f)));
            st6(Sout + 6 * qds, S0);
            st6(Sout + 6 * (qds + 1), S1);
            st6(Sout + 6 * (qds + 2), S2);
            v_j = S0 * jqd[qds] + S1 * jqd[qds + 1] + S2 * jqd[qds + 2];
        } else if (type == FJ_FREE || type == FJ_DISTANCE) {
            v_j = twist_xf(X_s, ld6(jqd + qds));
#pragma unroll
            for (int k = 0; k < 6; ++k) {
                S6 e;
                e.v[k] = 1.0f;
                st6(Sout + 6 * (qds + k), twist_xf(X_s, e));
            }
        }
        st6(sm.vs + 6 * child, v_j);
        st6(sm.as + 6 * child, c_app);
        st3(sm.so + 3 * child, solve_origin);
        const Xf X_sm = ldx(sm.bqc + 7 * child);
        spatial_inertia(Xf(X_sm.p - solve_origin, X_sm.q), d.body_mass[b0 + child], ldm(d.body_inertia + 9 * (b0 + child)), sm.Is + 36 * child);
    }
    __syncwarp(gmask);
    for (int lvl = 0; lvl <= M.max_depth; ++lvl) {  // B: v_s = v_parent + v_j, a_s = a_parent + v_s x v_j + c_app
        for (int j = l; j < nj; j += L) {
            const int gj = j0 + j;
            if (jdepth[gj] != lvl) continue;
            const int parent = jparent[gj], child = jchild[gj] - b0;
            const S6 v_j = ld6(sm.vs + 6 * child), c_app = ld6(sm.as + 6 * child);
            S6 v_par, a_par;
            if (parent >= 0) {
                v_par = ld6(sm.vs + 6 * (parent - b0));
                a_par = ld6(sm.as + 6 * (parent - b0));
            }
            const S6 v_s = v_par + v_j;
            const S6 a_s = a_par + scross(v_s, v_j) + c_app;
            st6(sm.vs + 6 * child, v_s);
            st6(sm.as + 6 * child, a_s);
        }
        __syncwarp(gmask);
    }
    for (int j = l; j < nj; j += L) {  // C: body forces
        const int gj = j0 + j, child = jchild[gj] - b0;
        const S6 v_s = ld6(sm.vs + 6 * child), a_s = ld6(sm.as + 6 * child);
        const V3 x_com_s = ld3(sm.bqc + 7 * child) - ld3(sm.so + 3 * child);
        const float mass = d.body_mass[b0 + child];
        int wi = d.body_world[b0 + child];
        if (wi < 0) wi += d.gravity_count;
        const V3 f_g = mass * ld3(d.gravity + 3 * wi);
        const S6 f_g_s(f_g, cross(x_com_s, f_g));
        const float* Is = sm.Is + 36 * child;
        const S6 f_b = m66v(Is, a_s) + scross_dual(v_s, m66v(Is, v_s));
        const V3 om = v_s.bot();
        const V3 v_com_world = v_s.top() + cross(om, x_com_s);
        st6(sm.qdfk + 6 * child, S6(v_com_world, om));
        st6(sm.fb + 6 * child, f_b - f_g_s);
    }
    __syncwarp(gmask);
    NB2_PHASE();
    // ---- eval_body_contact (penalty), ordered per body over the env's contacts ---------------------------
    // Two passes per chunk of contacts.  (A) one lane per CONTACT evaluates the penalty force once (the scan-per-body version made
    // every foot lane evaluate its ~4 contacts one after the other, each behind a chain of dependent global loads) and parks
    // (f_total, r_a x f_total, r_b x f_total, body pair) in a scratch record; (B) one lane per BODY adds its records in contact order,
    // side A before side B - the summation order of the reference's serial device, so the result is bit-identical.  The records
    // live in whichever dead block is larger: H (not formed yet) or v_s / a_s (dead between the RNEA forward pass and the closing FK).
    if (use_contacts) {
        constexpr int CR = 11;  // odd stride: lanes = consecutive contacts hit different banks
        const int cap_h = M.max_env_H / CR, cap_v = (12 * M.max_env_bodies) / CR;
        float* crec = cap_h >= cap_v ? sm.H : sm.vs;
        const int ccap = cap_h >= cap_v ? cap_h : cap_v;  // >= 1: an environment has at least one body
        for (int cbase = 0; cbase < nc; cbase += ccap) {
            const int cend = min(nc, cbase + ccap);
            for (int c = cbase + l; c < cend; c += L) {
                const int s = slot0 + c;
                const int ba = __float_as_int(cb[CF_BODY_A * T + s]), bb = __float_as_int(cb[CF_BODY_B * T + s]);
                float* rec = crec + (c - cbase) * CR;
                int code = 0;
                if (ba >= 0 || bb >= 0) {
                    const float ke = cb[CF_KE * T + s], kd = cb[CF_KD * T + s], kf = cb[CF_KF * T + s], ka = cb[CF_KA * T + s], mu = cb[CF_MU * T + s];
                    const V3 n = -V3(cb[CF_NX * T + s], cb[CF_NY * T + s], cb[CF_NZ * T + s]);
                    V3 bx_a(cb[CF_P0X * T + s], cb[CF_P0Y * T + s], cb[CF_P0Z * T + s]);
                    V3 bx_b(cb[CF_P1X * T + s], cb[CF_P1Y * T + s], cb[CF_P1Z * T + s]);
                    V3 r_a, r_b;
                    if (ba >= 0) {
                        const Xf X = ldx(sm.bq + 7 * ba);
                        bx_a = xpoint(X, bx_a) - cb[CF_MARGIN0 * T + s] * n;
                        r_a = bx_a - xpoint(X, ld3(d.body_com + 3 * (b0 + ba)));
                    }
                    if (bb >= 0) {
                        const Xf X = ldx(sm.bq + 7 * bb);
                        bx_b = xpoint(X, bx_b) + cb[CF_MARGIN1 * T + s] * n;
                        r_b = bx_b - xpoint(X, ld3(d.body_com + 3 * (b0 + bb)));
                    }
                    const float dd = dot(n, bx_a - bx_b);
                    if (dd < ka) {
                        V3 bv_a, bv_b;
                        if (ba >= 0) bv_a = ld3(sm.qdfk + 6 * ba) + cross(ld3(sm.qdfk + 6 * ba + 3), r_a);
                        if (bb >= 0) bv_b = ld3(sm.qdfk + 6 * bb) + cross(ld3(sm.qdfk + 6 * bb + 3), r_b);
                        const V3 v = bv_a - bv_b;
                        const float vn = dot(n, v);
                        const V3 vt = v - n * vn;
                        const float fn = dd * ke;
                        const float fd = fmin_w(vn, 0.0f) * kd * (dd < 0.0f ? 1.0f : 0.0f);
                        V3 ft;
                        if (dd < 0.0f) {
                            const float a2 = dot(vt, vt), delta = P.friction_smoothing;
                            const float vs = (a2 <= delta * delta) ? 0.5f * a2 : delta * (sqrtf(a2) - 0.5f * delta);
                            if (vs > 0.0f) {
                                const V3 fr = vt / vs;
                                ft = fr * fmin_w(kf * vs, -mu * (fn + fd));
                            }
                        }
                        const V3 f_total = n * (fn + fd) + ft;
                        st3(rec, f_total);
                        st3(rec + 3, cross(r_a, f_total));
                        st3(rec + 6, cross(r_b, f_total));
                        code = (ba + 1) | ((bb + 1) << 16);
                    }
                }
                reinterpret_cast<int*>(rec)[9] = code;  // 0 = no contribution (beyond the adhesion distance / no body)
            }
            __syncwarp(gmask);
            for (int b = l; b < nb; b += L) {
                V3 facc = ld3(sm.fe + 6 * b), tacc = ld3(sm.fe + 6 * b + 3);
                bool any = false;
                for (int c = 0; c < cend - cbase; ++c) {
                    const float* rec = crec + c * CR;
                    const int code = reinterpret_cast<const int*>(rec)[9];
                    const int ba = (code & 0xffff) - 1, bb = (code >> 16) - 1;
                    if (ba == b) { facc -= ld3(rec); tacc -= ld3(rec + 3); any = true; }
                    if (bb == b) { facc += ld3(rec); tacc += ld3(rec + 6); any = true; }
                }
                if (any) {
                    st3(sm.fe + 6 * b, facc);
                    st3(sm.fe + 6 * b + 3, tacc);
                }
            }
            __syncwarp(gmask);
        }
    }
    // zero_kinematic_body_forces (featherstone/kernels.py:55-63): a kinematic body ignores body_f, joint wrenches and contacts
    for (int b = l; b < nb; b += L)
        if (d.body_flags[b0 + b] & 2) st6(sm.fe + 6 * b, S6());
    __syncwarp(gmask);
    NB2_PHASE();
    // ---- eval_rigid_tau (RNEA backward).  The drive / limit / damping terms do not depend on the force recursion: they are
    // evaluated for all dofs at once and parked in tau[]; the level loop only adds -S.f_s in the reference's order. ---------
    for (int j = l; j < nj; j += L) {
        const int gj = j0 + j, type = jtype[gj];
        const int ds = jqds[gj], cs = jqs[gj], tqs = d.joint_target_q_start[gj];
        const int lin = jdim[2 * gj], ang = jdim[2 * gj + 1];
        const float* jqd = sm.qd_in - d0;
        float* tau = sm.tau - d0;
        if (type == FJ_BALL) {
            for (int k = 0; k < 3; ++k) tau[ds + k] = -d.joint_damping[ds + k] * jqd[ds + k];  // passive_f
        } else if (type == FJ_PRISMATIC || type == FJ_REVOLUTE || type == FJ_D6) {
            for (int k = 0; k < lin + ang; ++k) {
                const int jj = ds + k;
                tau[jj] = joint_force(sin.joint_q[cs + k], jqd[jj], ctl.joint_target_q[tqs + k], ctl.joint_target_qd[jj], d.joint_target_ke[jj],
                                      d.joint_target_kd[jj], d.joint_limit_lower[jj], d.joint_limit_upper[jj], d.joint_limit_ke[jj],
                                      d.joint_limit_kd[jj], d.joint_damping[jj]);
            }
        }
    }
    __syncwarp(gmask);
    for (int lvl = M.max_depth; lvl >= 0; --lvl) {
        for (int j = l; j < nj; j += L) {
            const int gj = j0 + j;
            if (jdepth[gj] != lvl) continue;
            const int type = jtype[gj], child = jchild[gj] - b0;
            const int ds = jqds[gj];
            const int lin = jdim[2 * gj], ang = jdim[2 * gj + 1];
            const S6 f_b = ld6(sm.fb + 6 * child), f_t = ld6(sm.ft + 6 * child), fe = ld6(sm.fe + 6 * child);
            const V3 x_com_s = ld3(sm.bqc + 7 * child) - ld3(sm.so + 3 * child);
            const S6 f_ext0(fe.top(), fe.bot() + cross(x_com_s, fe.top()));
            S6 f_ext;
#pragma unroll
            for (int k = 0; k < 6; ++k) f_ext.v[k] = -f_ext0.v[k];
            const S6 f_s = f_b + f_t + f_ext;
            st6(sm.fs + 6 * j, f_s);
            const float* S = sm.S - 6 * d0;
            const float* jf = sm.jf - d0;
            float* tau = sm.tau - d0;
            if (type == FJ_BALL) {
                for (int k = 0; k < 3; ++k) {
                    const int jj = ds + k;
                    tau[jj] = -dot6(ld6(S + 6 * jj), f_s) + jf[jj] + tau[jj];  // + passive_f
                }
            } else if (type == FJ_FREE || type == FJ_DISTANCE) {
                for (int k = 0; k < 6; ++k) tau[ds + k] = -dot6(ld6(S + 6 * (ds + k)), f_s) + jf[ds + k];
            } else if (type == FJ_PRISMATIC || type == FJ_REVOLUTE || type == FJ_D6) {
                for (int k = 0; k < lin + ang; ++k) {
                    const int jj = ds + k;
                    tau[jj] = -dot6(ld6(S + 6 * jj), f_s) + tau[jj] + jf[jj];  // + drive + joint_f
                }
            }
        }
        __syncwarp(gmask);
        // fold this level's f_s into the parents (serial reference order: descending joint index); the body's joint list is
        // ascending, so walk it backwards and take the joints it is the parent of
        for (int b = l; b < nb; b += L) {
            const int gb = b0 + b;
            S6 acc = ld6(sm.ft + 6 * b);
            bool any = false;
            for (int k = M.body_joint_start[gb + 1] - 1; k >= M.body_joint_start[gb]; --k) {
                const int e = M.body_joint_entry[k];
                if (e & 1) continue;  // the body is this joint's child
                const int j = e >> 1;
                if (jdepth[j0 + j] != lvl) continue;
                acc = acc + ld6(sm.fs + 6 * j);
                any = true;
            }
            if (any) st6(sm.ft + 6 * b, acc);
        }
        __syncwarp(gmask);
    }
    if constexpr (PF) {
        // ---- State.body_parent_f: the wrench the inbound joint transmits = this joint's RNEA backward-pass sum f_s (still in
        // sm.fs), moved from the solve origin to the child's COM; bodies without an inbound joint report zero ------------------
        for (int b = l; b < nb; b += L) st6(sout.body_parent_f + 6 * (b0 + b), S6());
        __syncwarp(gmask);
        for (int j = l; j < nj; j += L) {
            const int child = jchild[j0 + j] - b0;
            const S6 f_s = ld6(sm.fs + 6 * j);
            const V3 r_com = ld3(sm.bqc + 7 * child) - ld3(sm.so + 3 * child);
            st6(sout.body_parent_f + 6 * (b0 + child), S6(f_s.top(), f_s.bot() - cross(r_com, f_s.top())));
        }
        __syncwarp(gmask);
    }
    NB2_PHASE();
    // ---- H = J^T M J + Cholesky, per articulation -----------------------------------------------------------------
    if constexpr (TILE) {
        if (update_mass) {  // tensor-core path: the whole warp forms the H of each of its environments' articulations in turn
            __syncwarp();
            const size_t stride = fs_smem_floats(M);
            for (int g = 0; g < G; ++g) {
                const int env_g = (blockIdx.x * WARPS + warp) * G + g;
                if (env_g >= M.env_count) continue;  // warp-uniform
                const FsSmem sg = fs_carve(smem + size_t(warp * G + g) * stride, M);
                const int gj0 = M.env_joint_start[env_g], gb0 = M.env_body_start[env_g], gd0 = d.joint_qd_start[gj0];
                for (int art = M.env_art_start[env_g]; art < M.env_art_start[env_g + 1]; ++art) {
                    const int aj0 = d.articulation_start[art], aj1 = d.articulation_start[art + 1];
                    const int ad0 = d.joint_qd_start[aj0], n = d.joint_qd_start[aj1] - ad0;
                    // scratch: the v_s / a_s blocks (12 floats per body, dead until the closing FK rewrites them)
                    tile_mass_matrix(sg.S + 6 * (ad0 - gd0), sg.Is + 36 * (aj0 - gb0), M.joint_anc_mask + aj0, M.dof_joint + ad0, aj1 - aj0, n,
                                     sg.vs, sg.H + M.art_H_start[art]);
                }
            }
            __syncwarp();
        }
    }
    for (int a = 0; a < na; ++a) {
        const int art = a0 + a;
        const int aj0 = d.articulation_start[art], aj1 = d.articulation_start[art + 1];
        const int anj = aj1 - aj0;
        const int ad0 = jqds[aj0], n = jqds[aj1] - ad0;
        float* H = sm.H + M.art_H_start[art];
        float* Lg = M.fs_L + M.env_H_start[env] + M.art_H_start[art];
        if (update_mass) {
            // H = J^T (M J), lower triangle only (all dense_cholesky reads).  Columns are processed in batches of equal
            // (tree depth of their joint, dof index inside the joint): such joints are never ancestors of one another, so
            // every body lies below at most one of them and one 6-vector per body holds P[:, b] = I_i S_b for the whole batch:
            //   stage 1  P_i = I_i S_b           for the bodies below the batch's joints (one lane per body)
            //   stage 2  H[a, b] = sum_i sum_r S_a[r] P_i[r] over the bodies below joint(a), in (i, r) order, a >= b
            // - the summation order of the reference's dense_gemm pair (kernels.py:1504-1538) minus its exact-zero terms, so
            // the result is bit-identical while M J is formed once per column instead of once per entry.
            // The batch schedule is static topology: nb2_model_create tabulated, per batch, the column each body forms (hb_body_col)
            // and the column each row sums (hb_row_col); the kernel only indexes.  P is double-buffered (second copy in the dead
            // external-force block), so one group barrier per batch orders "P written" -> "P read" and the next batch's stage 1
            // overlaps the slow lanes' stage 2.
            if constexpr (!TILE) {
            for (int e = l; e < n * n; e += L) H[e] = 0.0f;
            const int nbatch = M.art_batch_count[art];
            const signed char* body_col = M.hb_body_col + M.art_hb_body_start[art];
            const signed char* row_col = M.hb_row_col + M.art_hb_row_start[art];
            const signed char* dofj = M.dof_joint + ad0;
            const float* Sart = sm.S + 6 * (ad0 - d0);
            // The schedule tables are per articulation, i.e. every environment reads its own copy: inside the batch loop each
            // lookup was a dependent global load (7 % of the stall samples, profiles/r2o_featherstone_step_kernel_hot_lines.txt).
            // They are staged once - row masks, then the two byte tables - in the dead v_s / a_s block when they fit.
            const int words_body = (nbatch * anj + 3) >> 2, words_row = (nbatch * n + 3) >> 2;
            const bool staged = 2 * n + words_body + words_row <= 12 * M.max_env_bodies;
            const unsigned long long* row_mask = nullptr;  // staged: descendant mask of the joint of dof `ra`
            if (staged) {
                unsigned long long* sm_mask = reinterpret_cast<unsigned long long*>(sm.vs);
                signed char* sm_body = reinterpret_cast<signed char*>(sm.vs + 2 * n);
                signed char* sm_row = sm_body + 4 * words_body;
                for (int i = l; i < n; i += L) sm_mask[i] = M.joint_desc_mask[aj0 + dofj[i]];
                for (int i = l; i < nbatch * anj; i += L) sm_body[i] = body_col[i];
                for (int i = l; i < nbatch * n; i += L) sm_row[i] = row_col[i];
                row_mask = sm_mask;
                body_col = sm_body;
                row_col = sm_row;
            }
            __syncwarp(gmask);
            for (int t = 0; t < nbatch; ++t) {
                float* Pb = (t & 1) ? sm.fe : sm.P;
                for (int i = l; i < anj; i += L) {  // stage 1: P_i = I_i S_col for the bodies below the batch's joints
                    const int col = body_col[t * anj + i];
                    if (col < 0) continue;
                    const S6 Sb = ld6(Sart + 6 * col);
                    // NB: the reference's spatial_mass indexes body_I_s by JOINT index (kernels.py:1476-1477)
                    const float* Is = sm.Is + 36 * (aj0 + i - b0);
#pragma unroll
                    for (int r = 0; r < 6; ++r) {
                        float pr = 0.0f;  // P[6i+r, b] = sum_k M[6i+r, 6i+k] J[6i+k, b]
#pragma unroll
                        for (int k = 0; k < 6; ++k) pr += Is[6 * r + k] * Sb.v[k];
                        Pb[6 * i + r] = pr;
                    }
                }
                __syncwarp(gmask);
                for (int ra = l; ra < n; ra += L) {  // stage 2: H[ra, col] over the bodies below joint(ra), ascending
                    const int col = row_col[t * n + ra];
                    if (col < 0) continue;
                    const S6 Sa = ld6(Sart + 6 * ra);
                    float sum = 0.0f;
                    for (unsigned long long m = staged ? row_mask[ra] : M.joint_desc_mask[aj0 + dofj[ra]]; m; m &= m - 1ull) {
                        const int i = __ffsll((long long)m) - 1;
#pragma unroll
                        for (int r = 0; r < 6; ++r) sum += Sa.v[r] * Pb[6 * i + r];
                    }
                    H[ra * n + col] = sum;
                }
            }
            }  // !TILE
            __syncwarp(gmask);
            // joint_armature_effective (solver_featherstone.py:269-281): 1e10 on the dofs of a joint driving a kinematic body.  The
            // reference adds it to the diagonal first thing in column jn; adding it here for all columns at once is the same sum
            // without a three-deep dependent global load in each of the n serial column steps.
            for (int i = l; i < n; i += L) {
                const bool kin_dof = (d.body_flags[jchild[aj0 + M.dof_joint[ad0 + i]]] & 2) != 0;
                H[i * n + i] = H[i * n + i] + (kin_dof ? 1.0e10f : d.joint_armature[ad0 + i]);
            }
            __syncwarp(gmask);
            // dense_cholesky (kernels.py:1690-1719), in place on the lower triangle; columns in order, rows in parallel.  Every lane
            // forms the pivot (same serial sum) next to its own row's entry of the column: the two subtraction chains are independent,
            // so they share one k loop and overlap.  The pivot is stored one step late - after the group barrier that ends its column -
            // because lanes still reading H[jn, jn] as the start of their own pivot sum must not see the square root.
            float pivot = 0.0f;
            for (int jn = 0; jn < n; ++jn) {
                if (l == 0 && jn > 0) H[(jn - 1) * n + (jn - 1)] = pivot;
                const int i0 = jn + 1 + l;
                float sdiag = H[jn * n + jn];
                float t = i0 < n ? H[i0 * n + jn] : 0.0f;
                for (int k = 0; k < jn; ++k) {
                    const float r = H[jn * n + k];
                    sdiag -= r * r;
                    if (i0 < n) t -= H[i0 * n + k] * r;
                }
                sdiag = sqrtf(sdiag);
                const float invS = 1.0f / sdiag;
                if (i0 < n) H[i0 * n + jn] = t * invS;
                for (int i = i0 + L; i < n; i += L) {  // more rows than lanes
                    float t2 = H[i * n + jn];
                    for (int k = 0; k < jn; ++k) t2 -= H[i * n + k] * H[jn * n + k];
                    H[i * n + jn] = t2 * invS;
                }
                pivot = sdiag;
                __syncwarp(gmask);
            }
            if (l == 0 && n > 0) H[(n - 1) * n + (n - 1)] = pivot;
            __syncwarp(gmask);
            for (int e = l; e < n * n; e += L) Lg[e] = H[e];
        } else {
            for (int e = l; e < n * n; e += L) H[e] = Lg[e];
        }
        __syncwarp(gmask);
        // dense_subs (kernels.py:1754-1781): forward then backward substitution, each row's subtractions in the serial loop's order
        {   // forward substitution, column-oriented: as soon as x[j] is final every later row subtracts L[i,j] x[j] - each row
            // still performs its subtractions in ascending j and divides last, i.e. the serial loop's arithmetic
            float* x = sm.qdd + (ad0 - d0);
            const float* bvec = sm.tau + (ad0 - d0);
            for (int i = l; i < n; i += L) x[i] = bvec[i];
            __syncwarp(gmask);
            for (int j = 0; j < n; ++j) {
                if (l == j % L) x[j] = x[j] / H[j * n + j];
                __syncwarp(gmask);
                const float xj = x[j];
                for (int i = j + 1 + ((l - (j + 1)) % L + L) % L; i < n; i += L) x[i] -= H[i * n + j] * xj;  // rows > j owned by this lane
            }
            __syncwarp(gmask);
        }
        // backward substitution: every row needs ALL later unknowns before its first (ascending-order) subtraction.  Shuffle-broadcast
        // substitutions with the backward products staged in the upper triangle were bit-exact but slower: 82.4 vs 80.3 us at 4096
        // quadruped envs (profiles/r2q_featherstone_subst_ab.txt)
        if (l == 0) {
            float* x = sm.qdd + (ad0 - d0);
            for (int i = n - 1; i >= 0; --i) {
                float t = x[i];
                for (int j = i + 1; j < n; ++j) t -= H[j * n + i] * x[j];
                x[i] = t / H[i * n + i];
            }
        }
        __syncwarp(gmask);
        for (int i = l; i < n; i += L)  // zero_kinematic_joint_qdd (kernels.py:1933-1948)
            if (d.body_flags[jchild[aj0 + M.dof_joint[ad0 + i]]] & 2) sm.qdd[ad0 - d0 + i] = 0.0f;
        __syncwarp(gmask);
    }
    NB2_PHASE();
    // ---- integrate_generalized_joints (jcalc_integrate, kernels.py:464-630) ----------------------------------------
    for (int j = l; j < nj; j += L) {
        const int gj = j0 + j, type = jtype[gj], parent = jparent[gj], child = jchild[gj];
        const int cs = jqs[gj], ds = jqds[gj];
        const float* q = sin.joint_q;
        const float* qd = sm.qd_in - d0;
        const float* qdd = sm.qdd - d0;
        float* qn = sm.jq - c0;
        float* qdn = sm.qd_out - d0;
        if (d.body_flags[child] & 2) {  // copy_kinematic_joint_state (kernels.py:1951-1976): the prescribed state passes through
            for (int i = cs; i < jqs[gj + 1]; ++i) qn[i] = q[i];
            for (int i = ds; i < jqds[gj + 1]; ++i) qdn[i] = qd[i];
            continue;
        }
        if (type == FJ_FIXED) continue;
        if (type == FJ_PRISMATIC || type == FJ_REVOLUTE) {
            const float qd_new = qd[ds] + qdd[ds] * dt;
            qdn[ds] = qd_new;
            qn[cs] = q[cs] + qd_new * dt;
        } else if (type == FJ_BALL) {
            const V3 w_new = V3(qd[ds], qd[ds + 1], qd[ds + 2]) + V3(qdd[ds], qdd[ds + 1], qdd[ds + 2]) * dt;
            const Q4 r(q[cs], q[cs + 1], q[cs + 2], q[cs + 3]);
            const Q4 drdt = qscale(qmul(Q4(w_new.x, w_new.y, w_new.z, 0.0f), r), 0.5f);
            const Q4 rn = qunit(qadd(r, qscale(drdt, dt)));
            qn[cs] = rn.x; qn[cs + 1] = rn.y; qn[cs + 2] = rn.z; qn[cs + 3] = rn.w;
            qdn[ds] = w_new.x; qdn[ds + 1] = w_new.y; qdn[ds + 2] = w_new.z;
        } else if (type == FJ_FREE || type == FJ_DISTANCE) {
            if (parent < 0) {
                const V3 a_parent(qdd[ds], qdd[ds + 1], qdd[ds + 2]), alpha(qdd[ds + 3], qdd[ds + 4], qdd[ds + 5]);
                const V3 v_parent(qd[ds], qd[ds + 1], qd[ds + 2]), omega(qd[ds + 3], qd[ds + 4], qd[ds + 5]);
                const V3 pp(q[cs], q[cs + 1], q[cs + 2]);
                const Q4 r(q[cs + 3], q[cs + 4], q[cs + 5], q[cs + 6]);
                const V3 r_com_joint = xpoint(xinv(ldx(d.joint_X_c + 7 * gj)), ld3(d.body_com + 3 * child));
                const V3 x_com = pp + qrot(r, r_com_joint);
                const V3 v_com = v_parent + cross(omega, x_com);
                const V3 a_com = a_parent + cross(alpha, x_com) + cross(omega, v_com);
                const V3 omega_new = omega + alpha * dt;
                const V3 v_com_new = v_com + a_com * dt;
                const Q4 drdt = qscale(qmul(Q4(omega_new.x, omega_new.y, omega_new.z, 0.0f), r), 0.5f);
                const Q4 r_new = qunit(qadd(r, qscale(drdt, dt)));
                const V3 x_com_new = x_com + v_com_new * dt;
                const V3 p_new = x_com_new - qrot(r_new, r_com_joint);
                const V3 v_parent_new = v_com_new - cross(omega_new, x_com_new);
                qn[cs] = p_new.x; qn[cs + 1] = p_new.y; qn[cs + 2] = p_new.z;
                qn[cs + 3] = r_new.x; qn[cs + 4] = r_new.y; qn[cs + 5] = r_new.z; qn[cs + 6] = r_new.w;
                qdn[ds] = v_parent_new.x; qdn[ds + 1] = v_parent_new.y; qdn[ds + 2] = v_parent_new.z;
                qdn[ds + 3] = omega_new.x; qdn[ds + 4] = omega_new.y; qdn[ds + 5] = omega_new.z;
            } else {
                const V3 w_s = V3(qd[ds + 3], qd[ds + 4], qd[ds + 5]) + V3(qdd[ds + 3], qdd[ds + 4], qdd[ds + 5]) * dt;
                const V3 v_s = V3(qd[ds], qd[ds + 1], qd[ds + 2]) + V3(qdd[ds], qdd[ds + 1], qdd[ds + 2]) * dt;
                const V3 p_s(q[cs], q[cs + 1], q[cs + 2]);
                const V3 dpdt = v_s + cross(w_s, p_s);
                const Q4 r_s(q[cs + 3], q[cs + 4], q[cs + 5], q[cs + 6]);
                const Q4 drdt = qscale(qmul(Q4(w_s.x, w_s.y, w_s.z, 0.0f), r_s), 0.5f);
                const V3 pn = p_s + dpdt * dt;
                const Q4 rn = qunit(qadd(r_s, qscale(drdt, dt)));
                qn[cs] = pn.x; qn[cs + 1] = pn.y; qn[cs + 2] = pn.z; qn[cs + 3] = rn.x; qn[cs + 4] = rn.y; qn[cs + 5] = rn.z; qn[cs + 6] = rn.w;
                qdn[ds] = v_s.x; qdn[ds + 1] = v_s.y; qdn[ds + 2] = v_s.z; qdn[ds + 3] = w_s.x; qdn[ds + 4] = w_s.y; qdn[ds + 5] = w_s.z;
            }
        } else if (type == FJ_D6) {
            const int cnt = jdim[2 * gj] + jdim[2 * gj + 1];
            for (int k = 0; k < cnt; ++k) {
                const float qd_new = qd[ds + k] + qdd[ds + k] * dt;
                qdn[ds + k] = qd_new;
                qn[cs + k] = q[cs + k] + qd_new * dt;
            }
        }
    }
    __syncwarp(gmask);
    for (int i = l; i < ncoord; i += L) sout.joint_q[c0 + i] = sm.jq[i];
    NB2_PHASE();
    // ---- eval_fk_with_velocity_conversion: level-parallel; reuses bq (poses) and vs (COM twists) ------------------------
    for (int lvl = 0; lvl <= M.max_depth; ++lvl) {
        for (int j = l; j < nj; j += L) {
            const int gj = j0 + j;
            if (jdepth[gj] != lvl) continue;
            const int type = jtype[gj], parent = jparent[gj], child = jchild[gj] - b0;
            const int qs = jqs[gj], qds = jqds[gj];
            const int lin = jdim[2 * gj], ang = jdim[2 * gj + 1];
            const float* jq = sm.jq - c0;
            const float* jqd = sm.qd_out - d0;
            const Xf X_j = joint_transform(d, type, qds, lin, ang, jq, qs);
            V3 vj_lin, vj_ang;
            if (type == FJ_PRISMATIC) vj_lin = ld3(d.joint_axis + 3 * qds) * jqd[qds];
            if (type == FJ_REVOLUTE) vj_ang = ld3(d.joint_axis + 3 * qds) * jqd[qds];
            if (type == FJ_BALL) vj_ang = V3(jqd[qds], jqd[qds + 1], jqd[qds + 2]);
            if (type == FJ_FREE || type == FJ_DISTANCE) {
                vj_lin = V3(jqd[qds], jqd[qds + 1], jqd[qds + 2]);
                vj_ang = V3(jqd[qds + 3], jqd[qds + 4], jqd[qds + 5]);
            }
            if (type == FJ_D6) {
                for (int k = 0; k < 3; ++k)
                    if (lin > k) vj_lin += ld3(d.joint_axis + 3 * (qds + k)) * jqd[qds + k];
                const int iq = qs + lin, iqd = qds + lin;
                if (ang == 1) vj_ang = jqd[iqd] * ld3(d.joint_axis + 3 * iqd);
                if (ang == 2) {
                    V3 w0, w1;
                    axes2(ld3(d.joint_axis + 3 * iqd), ld3(d.joint_axis + 3 * (iqd + 1)), jq[iq], w0, w1);
                    vj_ang = w0 * jqd[iqd] + w1 * jqd[iqd + 1];
                }
                if (ang == 3) {
                    V3 w0, w1, w2;
                    axes3(ld3(d.joint_axis + 3 * iqd), ld3(d.joint_axis + 3 * (iqd + 1)), ld3(d.joint_axis + 3 * (iqd + 2)), jq[iq], jq[iq + 1], w0, w1, w2);
                    vj_ang = w0 * jqd[iqd] + w1 * jqd[iqd + 1] + w2 * jqd[iqd + 2];
                }
            }
            Xf X_wpj = ldx(d.joint_X_p + 7 * gj);
            Xf X_wp;
            if (parent >= 0) {
                X_wp = ldx(sm.bq + 7 * (parent - b0));
                X_wpj = xmul(X_wp, X_wpj);
            }
            const Xf X_wcj = xmul(X_wpj, X_j);
            const Xf X_wc = xmul(X_wcj, xinv(ldx(d.joint_X_c + 7 * gj)));
            const V3 x_child = X_wc.p;
            V3 v_parent_origin, w_parent;
            if (parent >= 0) {
                const V3 pv = ld3(sm.vs + 6 * (parent - b0));
                w_parent = ld3(sm.vs + 6 * (parent - b0) + 3);
                v_parent_origin = cross(w_parent, x_child - xpoint(X_wp, ld3(d.body_com + 3 * parent))) + pv;
            }
            const V3 lin_w = xvec(X_wpj, vj_lin);
            V3 ang_w = xvec(X_wpj, vj_ang);
            V3 lin_o;
            if (type == FJ_FREE || type == FJ_DISTANCE) {
                const S6 vw = twist_xf(X_wpj, S6(vj_lin, vj_ang));
                lin_o = cross(vw.bot(), x_child) + vw.top();
                ang_w = vw.bot();
            } else {
                lin_o = lin_w + cross(ang_w, x_child - X_wcj.p);
            }
            const V3 v_o = v_parent_origin + lin_o, w_o = w_parent + ang_w;
            const V3 v_com = cross(w_o, xvec(X_wc, ld3(d.body_com + 3 * (b0 + child)))) + v_o;
            stx(sm.bq + 7 * child, X_wc);
            st6(sm.vs + 6 * child, S6(v_com, w_o));
            stx(sout.body_q + 7 * (b0 + child), X_wc);
            st6(sout.body_qd + 6 * (b0 + child), S6(v_com, w_o));
        }
        __syncwarp(gmask);
    }
    // ---- internal -> public joint_qd ------------------------------------------------------------------------------
    for (int j = l; j < nj; j += L) {
        const int gj = j0 + j, type = jtype[gj];
        const int qd0 = jqds[gj], qd1 = jqds[gj + 1];
        if (type != FJ_FREE && type != FJ_DISTANCE) {
            for (int i = qd0; i < qd1; ++i) sout.joint_qd[i] = sm.qd_out[i - d0];
            continue;
        }
        const int parent = jparent[gj], child = jchild[gj] - b0;
        Xf X_wpj = ldx(d.joint_X_p + 7 * gj);
        if (parent >= 0) X_wpj = xmul(ldx(sm.bq + 7 * (parent - b0)), X_wpj);
        const V3 x_com = xpoint(ldx(sm.bq + 7 * child), ld3(d.body_com + 3 * (b0 + child)));
        const V3 r = qrot_inv(X_wpj.q, x_com - X_wpj.p);
        const float* qi = sm.qd_out + (qd0 - d0);
        const V3 v_int(qi[0], qi[1], qi[2]), omega(qi[3], qi[4], qi[5]);
        const V3 v_com = v_int + cross(omega, r);
        float* o = sout.joint_qd + qd0;
        o[0] = v_com.x; o[1] = v_com.y; o[2] = v_com.z; o[3] = omega.x; o[4] = omega.y; o[5] = omega.z;
    }
}

template <int L, bool PF, int WARPS, bool TILE>
static nb2_status launch_fs_W(nb2_model* m, const nb2_featherstone_params& p, const nb2_state_view& in, const nb2_state_view& out,
                              const nb2_control_view& ctl, int use_contacts, int update_mass, float dt, cudaStream_t s) {
    const DevModel& M = m->dev;
    constexpr int NE = (32 / L) * WARPS;
    const int blocks = (M.env_count + NE - 1) / NE;
    const size_t smem = fs_smem_floats(M) * NE * sizeof(float);
    if (smem > 48 * 1024)
        NB2_CUDA_CHECK(cudaFuncSetAttribute(featherstone_step_kernel<L, PF, WARPS, TILE>, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem)));
    NB2_CUDA_CHECK(cudaFuncSetAttribute(featherstone_step_kernel<L, PF, WARPS, TILE>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    featherstone_step_kernel<L, PF, WARPS, TILE><<<blocks, 32 * WARPS, smem, s>>>(M, p, in, out, ctl, use_contacts, update_mass, dt);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

// warps per CTA: the largest compiled width the batch fills on every SM (see launch_xpbd_L), shared memory permitting
template <int L, bool PF>
static nb2_status launch_fs_LP(nb2_model* m, const nb2_featherstone_params& p, const nb2_state_view& in, const nb2_state_view& out,
                              const nb2_control_view& ctl, int use_contacts, int update_mass, float dt, cudaStream_t s) {
    const DevModel& M = m->dev;
    const size_t per_env = fs_smem_floats(M) * sizeof(float) * (32 / L);  // per warp
    if (per_env > 220 * 1024) {
        set_error("featherstone_step: environment too large for the fused shared-memory kernel");
        return NB2_ERR_CAPACITY;
    }
    const long long per_sm = warps_per_sm(m, L);
    int warps = per_sm <= 1 ? 1 : (per_sm <= 4 ? 4 : 14);
    if (warps >= 14 && per_env * 14 > 220 * 1024) warps = 4;
    if (warps >= 4 && warps < 14 && per_env * 4 > 220 * 1024) warps = 1;
    if (p.use_tile_gemm) {
        // the tensor-core variant is compiled for the plain step of the 16- and 32-lane layouts (what use_tile_gemm targets upstream:
        // one 18-dof articulation per world); anything else is refused instead of silently taking the FP32 path
        if constexpr (!PF && (L == 16 || L == 32)) {
            if (M.max_env_dofs > 24 || 12 * M.max_env_bodies < 6 * 24 || m->host.max_art_dofs > 24) {
                set_error("nb2_featherstone_step: use_tile_gemm needs articulations of at most 24 dofs (and >= 12 bodies of scratch per env)");
                return NB2_ERR_UNSUPPORTED;
            }
            if (warps >= 14) return launch_fs_W<L, PF, 14, true>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
            if (warps >= 4) return launch_fs_W<L, PF, 4, true>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
            return launch_fs_W<L, PF, 1, true>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
        } else {
            set_error("nb2_featherstone_step: use_tile_gemm is available for the plain step (no body_parent_f) of 16 / 32-lane layouts");
            return NB2_ERR_UNSUPPORTED;
        }
    }
    if (warps >= 14) return launch_fs_W<L, PF, 14, false>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
    if (warps >= 4) return launch_fs_W<L, PF, 4, false>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
    return launch_fs_W<L, PF, 1, false>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
}

template <int L>
static nb2_status launch_fs_L(nb2_model* m, const nb2_featherstone_params& p, const nb2_state_view& in, const nb2_state_view& out,
                              const nb2_control_view& ctl, int use_contacts, int update_mass, float dt, cudaStream_t s) {
    if (out.body_parent_f) return launch_fs_LP<L, true>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
    return launch_fs_LP<L, false>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
}

nb2_status launch_featherstone_step(nb2_model* m, const nb2_featherstone_params& p, const nb2_state_view& in, const nb2_state_view& out,
                                    const nb2_control_view& ctl, int use_contacts, float dt, cudaStream_t s) {
    const DevModel& M = m->dev;
    if (M.d.joint_count == 0) {
        set_error("nb2_featherstone_step: model has no joints (free rigid bodies need add_body(), which creates FREE joints)");
        return NB2_ERR_UNSUPPORTED;
    }
    if (!m->host.featherstone_supported) {
        set_error("nb2_featherstone_step: unsupported model: " + m->host.featherstone_reason);
        return NB2_ERR_UNSUPPORTED;
    }
    if (!in.body_q || !in.body_f || !in.joint_q || !in.joint_qd || !out.body_q || !out.body_qd || !out.joint_q || !out.joint_qd ||
        !ctl.joint_f || !ctl.joint_target_q || !ctl.joint_target_qd) {
        set_error("nb2_featherstone_step: state / control arrays are NULL");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    // state_in may be state_out (reference solver_featherstone.py:472): every group finishes reading its environment's inputs
    // (joint_q in the integration pass is the last) before it writes the outputs, and no group touches another environment.
    const int interval = p.update_mass_matrix_interval > 0 ? p.update_mass_matrix_interval : 1;
    const int update_mass = (m->featherstone_step_count % interval) == 0;
    m->featherstone_step_count += 1;
    switch (m->lanes_per_env) {
        case 8: return launch_fs_L<8>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
        case 16: return launch_fs_L<16>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
        default: return launch_fs_L<32>(m, p, in, out, ctl, use_contacts, update_mass, dt, s);
    }
}

// ---- public newton.eval_fk (sim/articulation.py:237-475) ------------------------------------------------------------------
// A set-up / reset call (example_basic_urdf.py:87; ArticulationView.eval_fk on the done worlds of an RL loop), not part of the
// substep loop.  fk_joint is one iteration of the reference's joint loop (eval_single_articulation_fk :237-418): it reads the
// parent's freshly written pose / twist and writes the child's.
__device__ __forceinline__ void fk_joint(const nb2_model_desc& d, int i, const float* __restrict__ joint_q, const float* __restrict__ joint_qd,
                                         float* body_q, float* body_qd, int body_flag_filter) {
    const int type = d.joint_type[i], parent = d.joint_parent[i], child = d.joint_child[i];
    const int qs = d.joint_q_start[i], qds = d.joint_qd_start[i];
    const int lin = d.joint_dof_dim[2 * i], ang = d.joint_dof_dim[2 * i + 1];
    const Xf X_j = joint_transform(d, type, qds, lin, ang, joint_q, qs);
    V3 vj_lin, vj_ang;
    if (type == FJ_PRISMATIC) vj_lin = ld3(d.joint_axis + 3 * qds) * joint_qd[qds];
    if (type == FJ_REVOLUTE) vj_ang = ld3(d.joint_axis + 3 * qds) * joint_qd[qds];
    if (type == FJ_BALL) vj_ang = V3(joint_qd[qds], joint_qd[qds + 1], joint_qd[qds + 2]);
    if (type == FJ_FREE || type == FJ_DISTANCE) {
        vj_lin = V3(joint_qd[qds], joint_qd[qds + 1], joint_qd[qds + 2]);
        vj_ang = V3(joint_qd[qds + 3], joint_qd[qds + 4], joint_qd[qds + 5]);
    }
    if (type == FJ_D6) {
        for (int k = 0; k < 3; ++k)
            if (lin > k) vj_lin += ld3(d.joint_axis + 3 * (qds + k)) * joint_qd[qds + k];
        const int iq = qs + lin, iqd = qds + lin;
        if (ang == 1) vj_ang = joint_qd[iqd] * ld3(d.joint_axis + 3 * iqd);
        if (ang == 2) {
            V3 w0, w1;
            axes2(ld3(d.joint_axis + 3 * iqd), ld3(d.joint_axis + 3 * (iqd + 1)), joint_q[iq], w0, w1);
            vj_ang = w0 * joint_qd[iqd] + w1 * joint_qd[iqd + 1];
        }
        if (ang == 3) {
            V3 w0, w1, w2;
            axes3(ld3(d.joint_axis + 3 * iqd), ld3(d.joint_axis + 3 * (iqd + 1)), ld3(d.joint_axis + 3 * (iqd + 2)), joint_q[iq], joint_q[iq + 1],
                  w0, w1, w2);
            vj_ang = w0 * joint_qd[iqd] + w1 * joint_qd[iqd + 1] + w2 * joint_qd[iqd + 2];
        }
    }
    Xf X_wpj = ldx(d.joint_X_p + 7 * i);
    Xf X_wp;
    if (parent >= 0) {
        X_wp = ldx(body_q + 7 * parent);
        X_wpj = xmul(X_wp, X_wpj);
    }
    const Xf X_wcj = xmul(X_wpj, X_j);
    const Xf X_wc = xmul(X_wcj, xinv(ldx(d.joint_X_c + 7 * i)));
    const V3 x_child = X_wc.p;
    V3 v_parent_origin, w_parent;
    if (parent >= 0) {
        const V3 pv = ld3(body_qd + 6 * parent);
        w_parent = ld3(body_qd + 6 * parent + 3);
        v_parent_origin = cross(w_parent, x_child - xpoint(X_wp, ld3(d.body_com + 3 * parent))) + pv;
    }
    const V3 lin_w = xvec(X_wpj, vj_lin), ang_w = xvec(X_wpj, vj_ang);
    const V3 com_c = xvec(X_wc, ld3(d.body_com + 3 * child));
    V3 lin_o;
    if (type == FJ_FREE || type == FJ_DISTANCE) lin_o = lin_w - cross(ang_w, com_c);  // COM twist -> origin twist
    else lin_o = lin_w + cross(ang_w, x_child - X_wcj.p);
    const V3 v_o = v_parent_origin + lin_o, w_o = w_parent + ang_w;
    const V3 v_com = cross(w_o, com_c) + v_o;
    // body_flag_filter (sim/articulation.py:254, 421): a body whose flags miss the filter keeps its values; descendants read them
    if ((d.body_flags[child] & body_flag_filter) == 0) return;
    stx(body_q + 7 * child, X_wc);
    st6(body_qd + 6 * child, S6(v_com, w_o));
}

// Which articulation a work item handles: `mask` / `indices` are the reference's optional articulation_mask /
// articulation_indices (eval_articulation_fk :420-475); -1 = nothing to do.
__device__ __forceinline__ int fk_articulation(const nb2_model_desc& d, int item, int count, const uint8_t* mask, const int* indices) {
    if (item >= count) return -1;
    const int a = indices ? indices[item] : item;
    if (a < 0 || a >= d.articulation_count) return -1;
    if (mask && !mask[a]) return -1;
    return a;
}

// One WARP per articulation, joints of equal tree depth in parallel (lane = joint), depth levels in order with __syncwarp()
// between them (it orders the lanes' global writes and reads): a 13-joint quadruped takes 4 dependent steps instead of 13.
// Every joint runs exactly the arithmetic of the serial walk on the same parent values, so the results are bit-identical to it.
// Requires parent-before-child joint order and one driving joint per body (nb2_model::fk_levels, checked at model creation).
__global__ void __launch_bounds__(128) eval_fk_levels_kernel(DevModel M, const float* __restrict__ joint_q, const float* __restrict__ joint_qd,
                                                             float* body_q, float* body_qd, const uint8_t* __restrict__ mask,
                                                             const int* __restrict__ indices, int count, int body_flag_filter) {
    const nb2_model_desc& d = M.d;
    const int lane = threadIdx.x & 31;
    const int a = fk_articulation(d, (blockIdx.x * blockDim.x + threadIdx.x) >> 5, count, mask, indices);  // warp-uniform
    if (a < 0) return;
    const int j0 = d.articulation_start[a], j1 = d.articulation_start[a + 1];
    int deepest = 0;
    for (int i = j0 + lane; i < j1; i += 32) deepest = max(deepest, M.joint_depth[i]);
    for (int o = 16; o > 0; o >>= 1) deepest = max(deepest, __shfl_xor_sync(0xffffffffu, deepest, o));
    for (int level = 0; level <= deepest; ++level) {
        for (int i = j0 + lane; i < j1; i += 32)
            if (M.joint_depth[i] == level && d.joint_articulation[i] != -1) fk_joint(d, i, joint_q, joint_qd, body_q, body_qd, body_flag_filter);
        __syncwarp();
    }
}

// Fallback for models whose joint order the level schedule cannot honour: one thread walks one articulation in joint order.
__global__ void __launch_bounds__(128) eval_fk_kernel(DevModel M, const float* __restrict__ joint_q, const float* __restrict__ joint_qd,
                                                      float* body_q, float* body_qd, const uint8_t* __restrict__ mask,
                                                      const int* __restrict__ indices, int count, int body_flag_filter) {
    const nb2_model_desc& d = M.d;
    const int a = fk_articulation(d, blockIdx.x * blockDim.x + threadIdx.x, count, mask, indices);
    if (a < 0) return;
    for (int i = d.articulation_start[a]; i < d.articulation_start[a + 1]; ++i)
        if (d.joint_articulation[i] != -1) fk_joint(d, i, joint_q, joint_qd, body_q, body_qd, body_flag_filter);
}

nb2_status launch_eval_fk(nb2_model* m, const float* joint_q, const float* joint_qd, float* body_q, float* body_qd, cudaStream_t s,
                          const uint8_t* mask, const int* indices, int index_count, int body_flag_filter) {
    const int A = indices ? index_count : m->dev.d.articulation_count;
    if (A <= 0 || m->dev.d.articulation_count == 0) return NB2_OK;
    if (m->host.fk_levels)
        eval_fk_levels_kernel<<<(A + 3) / 4, 128, 0, s>>>(m->dev, joint_q, joint_qd, body_q, body_qd, mask, indices, A, body_flag_filter);
    else
        eval_fk_kernel<<<(A + 127) / 128, 128, 0, s>>>(m->dev, joint_q, joint_qd, body_q, body_qd, mask, indices, A, body_flag_filter);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

// ---- public newton.eval_ik (sim/articulation.py:640-932 eval_articulation_ik): one thread per joint -----------------------------
NB2_DEV float twist_angle_signed(V3 axis, Q4 q) {  // wp.quat_twist_angle_signed: 2 atan2(q.xyz . axis, q.w), range (-2 pi, 2 pi]
    return 2.0f * atan2_w(dot(V3(q.x, q.y, q.z), axis), q.w);
}

// newton.math.quat_decompose (math/spatial.py:150-175): wp.quat_to_euler(q, 2, 1, 0), each angle wrapped to [-pi, pi); for
// q = qx(a) qy(b) qz(c) the result is (a, b, c)
NB2_DEV float wrap_pm_pi(float theta) {
    const float pi = 3.14159265358979323846f, two_pi = 2.0f * pi;
    float wrapped = fmodf(theta + pi, two_pi);
    if (wrapped < 0.0f) wrapped += two_pi;
    return wrapped - pi;
}
NB2_DEV V3 q_decompose(Q4 q) {
    const float a = q.w - q.y, b = q.z - q.x, c = q.y + q.w, d = -q.x - q.z;
    const float n_ab = a * a + b * b;
    float theta2 = acos_w(2.0f * n_ab / (n_ab + c * c + d * d) - 1.0f);
    const float theta_plus = atan2_w(b, a), theta_minus = atan2_w(d, c);
    const float theta1 = theta_plus - theta_minus;
    float theta3 = theta_plus + theta_minus;
    theta3 = -theta3;
    theta2 -= 1.57079632679489661923f;
    return V3(wrap_pm_pi(theta3), wrap_pm_pi(theta2), wrap_pm_pi(theta1));
}
// invert_2d / invert_3d_rotational_dofs (sim/articulation.py:85-126, 177-236); `three` selects the 3-axis variant
NB2_DEV void invert_rotational_dofs(bool three, V3 axis_0, V3 axis_1, V3 axis_2, Q4 q_p, Q4 q_c, V3 w_err, float* angles_out, float* vel_out) {
    const V3 axis_2_rh = cross(axis_0, axis_1);
    float s = 1.0f;
    if (three && dot(axis_2_rh, axis_2) < 0.0f) s = -1.0f;
    const Q4 q_off = q_from_cols(axis_0, axis_1, axis_2_rh);
    const Q4 q_pc = qmul(qmul(qmul(qconj(q_off), qconj(q_p)), q_c), q_off);
    const V3 angles = q_decompose(q_pc);
    const V3 l0 = qrot(q_off, V3(1.f, 0.f, 0.f)), l1 = qrot(q_off, V3(0.f, 1.f, 0.f)), l2 = qrot(q_off, V3(0.f, 0.f, 1.f));
    const V3 a0 = l0;
    const Q4 q_0 = q_axis_angle(a0, angles.x);
    const V3 a1 = qrot(q_0, l1);
    const Q4 q_1 = q_axis_angle(a1, angles.y);
    const V3 a2 = qrot(qmul(q_1, q_0), l2);
    const V3 w_err_p = qrot_inv(q_p, w_err);
    const V3 c12 = cross(a1, a2), c02 = cross(a0, a2), c01 = cross(a0, a1);
    angles_out[0] = angles.x;
    angles_out[1] = angles.y;
    vel_out[0] = dot(w_err_p, c12) / dot(a0, c12);
    vel_out[1] = dot(w_err_p, c02) / dot(a1, c02);
    if (three) {
        angles_out[2] = s * angles.z;
        vel_out[2] = s * (dot(w_err_p, c01) / dot(a2, c01));
    }
}

__global__ void __launch_bounds__(128) eval_ik_kernel(DevModel M, const float* __restrict__ body_q, const float* __restrict__ body_qd,
                                                      float* __restrict__ joint_q, float* __restrict__ joint_qd) {
    const nb2_model_desc& d = M.d;
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= d.joint_count || d.joint_articulation[j] < 0) return;
    const int parent = d.joint_parent[j], child = d.joint_child[j], type = d.joint_type[j];
    const Xf X_pj = ldx(d.joint_X_p + 7 * j), X_cj = ldx(d.joint_X_c + 7 * j);
    V3 w_p, v_p, pv, pw;
    Xf X_wpj = X_pj, X_wp;
    if (parent >= 0) {
        X_wp = ldx(body_q + 7 * parent);
        X_wpj = xmul(X_wp, X_pj);
        pv = ld3(body_qd + 6 * parent);
        pw = ld3(body_qd + 6 * parent + 3);
        w_p = pw;
        v_p = cross(pw, X_wpj.p - xpoint(X_wp, ld3(d.body_com + 3 * parent))) + pv;
    }
    const Xf X_wc = ldx(body_q + 7 * child);
    const Xf X_wcj = xmul(X_wc, X_cj);
    const V3 cv = ld3(body_qd + 6 * child), w_c = ld3(body_qd + 6 * child + 3);
    const V3 v_c = cross(w_c, X_wcj.p - xpoint(X_wc, ld3(d.body_com + 3 * child))) + cv;
    const V3 x_err = X_wcj.p - X_wpj.p, v_err = v_c - v_p, w_err = w_c - w_p;
    const Q4 q_p = X_wpj.q, q_c = X_wcj.q;
    const int q_start = d.joint_q_start[j], qd_start = d.joint_qd_start[j];
    const int lin = d.joint_dof_dim[2 * j], ang = d.joint_dof_dim[2 * j + 1];
    if (type == FJ_PRISMATIC) {
        const V3 axis_p = qrot(q_p, ld3(d.joint_axis + 3 * qd_start));
        joint_q[q_start] = dot(x_err, axis_p);
        joint_qd[qd_start] = dot(v_err, axis_p);
    } else if (type == FJ_REVOLUTE) {
        const Q4 q_pc = qmul(qconj(q_p), q_c);
        const V3 ax = ld3(d.joint_axis + 3 * qd_start);
        joint_q[q_start] = twist_angle_signed(ax, q_pc);
        joint_qd[qd_start] = dot(w_err, xvec(X_wpj, ax));
    } else if (type == FJ_BALL) {
        const Q4 q_pc = qmul(qconj(q_p), q_c);
        joint_q[q_start] = q_pc.x; joint_q[q_start + 1] = q_pc.y; joint_q[q_start + 2] = q_pc.z; joint_q[q_start + 3] = q_pc.w;
        const V3 av = xvec(xinv(X_wpj), w_err);
        st3(joint_qd + qd_start, av);
    } else if (type == FJ_FREE || type == FJ_DISTANCE) {
        const Q4 q_pc = qmul(qconj(q_p), q_c);
        const V3 x_err_c = qrot_inv(q_p, x_err);
        const V3 x_com_w = xpoint(X_wc, ld3(d.body_com + 3 * child));
        V3 v_com_err = cv;
        if (parent >= 0) v_com_err = v_com_err - (cross(pw, x_com_w - xpoint(X_wp, ld3(d.body_com + 3 * parent))) + pv);
        const V3 v_err_c = qrot_inv(q_p, v_com_err), w_err_c = qrot_inv(q_p, w_err);
        st3(joint_q + q_start, x_err_c);
        joint_q[q_start + 3] = q_pc.x; joint_q[q_start + 4] = q_pc.y; joint_q[q_start + 5] = q_pc.z; joint_q[q_start + 6] = q_pc.w;
        st3(joint_qd + qd_start, v_err_c);
        st3(joint_qd + qd_start + 3, w_err_c);
    } else if (type == FJ_D6) {
        const V3 x_err_c = qrot_inv(q_p, x_err), v_err_c = qrot_inv(q_p, v_err);
        for (int k = 0; k < 3; ++k)
            if (lin > k) {
                const V3 ax = ld3(d.joint_axis + 3 * (qd_start + k));
                joint_q[q_start + k] = dot(x_err_c, ax);
                joint_qd[qd_start + k] = dot(v_err_c, ax);
            }
        if (ang == 1) {
            const Q4 q_pc = qmul(qconj(q_p), q_c);
            const V3 ax = ld3(d.joint_axis + 3 * (qd_start + lin));
            joint_q[q_start + lin] = twist_angle_signed(ax, q_pc);
            joint_qd[qd_start + lin] = dot(w_err, xvec(X_wpj, ax));
        }
        if (ang >= 2) {
            const int ia = qd_start + lin;
            invert_rotational_dofs(ang == 3, ld3(d.joint_axis + 3 * ia), ld3(d.joint_axis + 3 * (ia + 1)),
                                   ang == 3 ? ld3(d.joint_axis + 3 * (ia + 2)) : V3(), q_p, q_c, w_err, joint_q + q_start + lin, joint_qd + qd_start + lin);
        }
    }
}

nb2_status launch_eval_ik(nb2_model* m, const float* body_q, const float* body_qd, float* joint_q, float* joint_qd, cudaStream_t s) {
    const int J = m->dev.d.joint_count;
    if (J == 0) return NB2_OK;
    eval_ik_kernel<<<(J + 127) / 128, 128, 0, s>>>(m->dev, body_q, body_qd, joint_q, joint_qd);
    count_launch();
    NB2_CUDA_CHECK(cudaGetLastError());
    return NB2_OK;
}

}  // namespace nb2
