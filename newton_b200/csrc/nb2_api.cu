// nb2_api.cu - C-ABI entry points of libnewton_b200.so (include/newton_b200.h) and model ingestion.
//
// nb2_model_create() derives, once, the tables the fused per-environment kernels need from the reference-layout
// Model arrays: the env partition (worlds are contiguous index ranges: reference sim/model.py:1081-1097), the
// per-env explicit pair lists re-ordered by the deterministic contact key (reference geometry/contact_data.py:59-87),
// the per-body joint adjacency used for ordered (atomic-free) Jacobi accumulation, and the env-major contact blocks.
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <mutex>

#include <cmath>

#include "nb2_internal.cuh"

namespace nb2 {

static thread_local std::string g_last_error;
static std::atomic<int64_t> g_launches{0};

void set_error(const std::string& msg) { g_last_error = msg; }
void count_launch(int n) { g_launches.fetch_add(n, std::memory_order_relaxed); }

template <typename T>
static nb2_status fetch(const T* dptr, size_t n, std::vector<T>& out) {
    out.resize(n);
    if (n == 0) return NB2_OK;
    if (!dptr) {
        set_error("nb2_model_create: required model array is NULL");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    NB2_CUDA_CHECK(cudaMemcpy(out.data(), dptr, n * sizeof(T), cudaMemcpyDefault));
    return NB2_OK;
}

template <typename T>
static nb2_status upload(nb2_model* m, const std::vector<T>& v, const T** out) {
    void* p = nullptr;
    size_t bytes = std::max<size_t>(v.size(), 1) * sizeof(T);
    NB2_CUDA_CHECK(cudaMalloc(&p, bytes));
    m->allocations.push_back(p);
    if (!v.empty()) NB2_CUDA_CHECK(cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    *out = static_cast<const T*>(p);
    return NB2_OK;
}

static int pow2_at_least(int x) {
    int p = 1;
    while (p < x) p <<= 1;
    return p;
}

static nb2_status build_tables(nb2_model* m, const nb2_model_desc& d) {
    HostTables& h = m->host;
    const int W = d.world_count, B = d.body_count, J = d.joint_count, S = d.shape_count, P = d.shape_pair_count;
    if (W <= 0 || B < 0 || J < 0 || S < 0 || P < 0) {
        set_error("nb2_model_create: invalid counts");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    std::vector<int> bws, jws, sws, shape_world, shape_type, shape_body, jparent, jchild, pairs, art_start, jart;
    nb2_status st;
    if ((st = fetch(d.body_world_start, size_t(W) + 2, bws))) return st;
    if ((st = fetch(d.joint_world_start, size_t(W) + 2, jws))) return st;
    if ((st = fetch(d.shape_world_start, size_t(W) + 2, sws))) return st;
    if ((st = fetch(d.shape_world, size_t(S), shape_world))) return st;
    if ((st = fetch(d.shape_type, size_t(S), shape_type))) return st;
    if ((st = fetch(d.shape_body, size_t(S), shape_body))) return st;
    if ((st = fetch(d.joint_parent, size_t(J), jparent))) return st;
    if ((st = fetch(d.joint_child, size_t(J), jchild))) return st;
    if ((st = fetch(d.shape_contact_pairs, size_t(P) * 2, pairs))) return st;
    if ((st = fetch(d.articulation_start, size_t(d.articulation_count) + 1, art_start))) return st;
    if ((st = fetch(d.joint_articulation, size_t(J), jart))) return st;
    std::vector<float> shape_scale;
    if ((st = fetch(d.shape_scale, size_t(S) * 3, shape_scale))) return st;

    // ---- env partition ----------------------------------------------------------------------
    const bool implicit_single = (W == 1) && (bws[0] == B) && (jws[0] == J) && (sws[0] == S);
    m->implicit_single = implicit_single;
    int E;
    h.global_shapes.clear();
    if (implicit_single) {  // model built without begin_world(): everything lives in world -1 (builder.py:11276)
        E = 1;
        h.env_body_start = {0, B};
        h.env_joint_start = {0, J};
        h.env_shape_start = {0, S};
    } else {
        if (bws[0] != 0 || bws[W] != B || jws[0] != 0 || jws[W] != J) {
            set_error("bodies/joints in the global world (-1) of a multi-world model are not supported by the fused kernels");
            return NB2_ERR_UNSUPPORTED;
        }
        E = W;
        h.env_body_start.assign(bws.begin(), bws.begin() + W + 1);
        h.env_joint_start.assign(jws.begin(), jws.begin() + W + 1);
        h.env_shape_start.assign(sws.begin(), sws.begin() + W + 1);
        for (int s = 0; s < sws[0]; ++s) h.global_shapes.push_back(s);
        for (int s = sws[W]; s < S; ++s) h.global_shapes.push_back(s);
        for (int s : h.global_shapes)
            if (shape_body[s] != -1) {
                set_error("global (world -1) shapes must be static (body == -1)");
                return NB2_ERR_UNSUPPORTED;
            }
    }
    // articulations per env (articulations are world-contiguous like joints)
    h.env_art_start.assign(size_t(E) + 1, 0);
    {
        int a = 0;
        for (int e = 0; e < E; ++e) {
            h.env_art_start[e] = a;
            while (a < d.articulation_count && art_start[a] < h.env_joint_start[e + 1]) ++a;
        }
        h.env_art_start[E] = d.articulation_count;
    }
    auto env_of_shape = [&](int s) -> int {
        if (implicit_single) return 0;
        return shape_world[s];
    };
    std::vector<int> hull_count;
    {
        bool any_mesh = false;
        for (int s = 0; s < S; ++s) any_mesh = any_mesh || shape_type[s] == 8;
        if (any_mesh) {
            if (!d.hull_points || !d.shape_hull_start || !d.shape_hull_count) {
                set_error("MESH shapes need model.hull_points / shape_hull_start / shape_hull_count (the mesh vertex pool)");
                return NB2_ERR_INVALID_ARGUMENT;
            }
            if ((st = fetch(d.shape_hull_count, size_t(S), hull_count))) return st;
        }
    }
    m->has_mesh_pairs = false;
    // ---- pairs: group by env, order shapes by type, sort by the deterministic contact key ----
    struct PairRec { int env; int64_t key; int sa, sb; int max_contacts; };
    std::vector<PairRec> recs;
    recs.reserve(P);
    for (int t = 0; t < P; ++t) {
        int s1 = pairs[2 * t], s2 = pairs[2 * t + 1];
        if (s1 < 0 || s2 < 0 || s1 >= S || s2 >= S || s1 == s2) continue;
        int w1 = env_of_shape(s1), w2 = env_of_shape(s2);
        int env = w1 >= 0 ? w1 : w2;
        if (w1 >= 0 && w2 >= 0 && w1 != w2) continue;  // cross-world pairs never collide
        if (env < 0) continue;                           // static-vs-static global pair: no dynamic body involved
        int sa = s1, sb = s2, pair_max = 5;
        if (shape_type[sa] > shape_type[sb]) std::swap(sa, sb);  // narrow_phase.py:525-528
        {   // shapes the narrow phase of this library covers: analytic primitives + convex primitives through MPR/GJK
            const int ta = shape_type[sa], tb = shape_type[sb];
            // PLANE SPHERE CAPSULE ELLIPSOID CYLINDER BOX CONE CONVEX_MESH
            auto known = [](int t) { return t == 1 || (t >= 3 && t <= 10); };  // 8 = MESH (plane route only, below)
            if (!known(ta) || !known(tb)) {
                set_error("shape pair (" + std::to_string(sa) + "," + std::to_string(sb) + "): geometry types " + std::to_string(ta) + "/" +
                          std::to_string(tb) + " are outside the supported set (plane, sphere, capsule, ellipsoid, cylinder, box, cone, "
                          "convex mesh)");
                return NB2_ERR_UNSUPPORTED;
            }
            if ((ta == 10 || tb == 10) &&
                (!d.hull_points || !d.shape_hull_start || !d.shape_hull_count || !d.shape_collision_aabb_lower || !d.shape_collision_aabb_upper)) {
                set_error("CONVEX_MESH shapes need model.hull_points / shape_hull_start / shape_hull_count / shape_collision_aabb_lower / _upper");
                return NB2_ERR_INVALID_ARGUMENT;
            }
            if (ta == 8 || tb == 8) {  // mesh routing (narrow_phase.py:594-640)
                const bool infinite_plane_a = ta == 1 && shape_scale[3 * sa] == 0.0f && shape_scale[3 * sa + 1] == 0.0f;
                if (!(infinite_plane_a && tb == 8)) {
                    set_error("shape pair (" + std::to_string(sa) + "," + std::to_string(sb) + "): a MESH shape collides with infinite planes "
                              "only (one contact per vertex); mesh-mesh / mesh-convex / mesh-finite-plane need the reference's BVH / SDF "
                              "routes, which are out of scope - filter the pair or use a convex hull");
                    return NB2_ERR_UNSUPPORTED;
                }
                // narrow_phase.py:628: the pair is stored (mesh, plane) - shape_a of its contacts and of their sort key is the mesh
                m->has_mesh_pairs = true;
                recs.push_back({env, ((int64_t(sb) & 0xFFFFF) << 43) | ((int64_t(sa) & 0xFFFFF) << 23), sb, sa, hull_count[sb]});
                continue;
            }
            {   // narrow_phase.py:642-655 + the analytic chain of narrow_phase.py:657-864: everything else is MPR / GJK
                // (a plane that gets there - cone, barrel cylinder lying on its side - is replaced by a box proxy)
                const bool early = ta >= 5 || tb == 9 || (ta == 4 && tb > 4);
                const bool barrel = tb == 6 && shape_scale[3 * sb + 2] != 0.0f;
                const bool analytic = !early && ((ta == 1 && (tb == 3 || tb == 4 || tb == 5 || (tb == 6 && !barrel) || tb == 7)) ||
                                                 (ta == 3 && (tb == 3 || tb == 4 || tb == 7 || (tb == 6 && !barrel))) || (ta == 4 && tb == 4));
                if (!analytic) m->has_convex_pairs = true;
                pair_max = analytic ? 4 : 5;  // analytic colliders return <= 4 points (plane-box / plane-cylinder), manifolds <= 5
            }
        }
        int64_t key = ((int64_t(sa) & 0xFFFFF) << 43) | ((int64_t(sb) & 0xFFFFF) << 23);
        recs.push_back({env, key, sa, sb, pair_max});
    }
    std::stable_sort(recs.begin(), recs.end(), [](const PairRec& a, const PairRec& b) {
        return a.env != b.env ? a.env < b.env : a.key < b.key;
    });
    h.env_pair_start.assign(size_t(E) + 1, 0);
    h.env_slot_start.assign(size_t(E) + 1, 0);
    h.pairs.clear();
    h.pairs.reserve(recs.size());
    {
        size_t i = 0;
        for (int e = 0; e < E; ++e) {
            h.env_pair_start[e] = int(h.pairs.size());
            const int ss = h.env_shape_start[e], se = h.env_shape_start[e + 1];
            const int nloc = se - ss;
            auto slot_of = [&](int s) -> int {
                if (s >= ss && s < se) return s - ss;
                for (size_t g = 0; g < h.global_shapes.size(); ++g)
                    if (h.global_shapes[g] == s) return nloc + int(g);
                return -1;
            };
            int env_max = 0, env_slots = 0;
            for (; i < recs.size() && recs[i].env == e; ++i) {
                env_max += recs[i].max_contacts;
                m->max_env_contacts = std::max(m->max_env_contacts, env_max);
                int a = slot_of(recs[i].sa), b = slot_of(recs[i].sb);
                if (a < 0 || b < 0) {
                    set_error("contact pair references a shape outside its world");
                    return NB2_ERR_INVALID_ARGUMENT;
                }
                const bool mesh_pair = shape_type[recs[i].sa] == 8;  // (mesh, plane): flagged for the collide kernel
                h.pairs.push_back(make_int2(a, mesh_pair ? (b | NB2_PAIR_MESH_PLANE) : b));
                env_slots += mesh_pair ? recs[i].max_contacts : 5;
            }
            h.env_slot_start[e + 1] = h.env_slot_start[e] + env_slots;
        }
        h.env_pair_start[E] = int(h.pairs.size());
        h.explicit_env_slot_start = h.env_slot_start;
    }
    // (contact-block slot ranges: 5 slots per pair - <= 4 analytic, <= 5 manifold contacts - and one per vertex of a mesh-plane pair)
    // ---- per-body joint adjacency in joint order (parent entry before child entry of the same joint) ----
    h.body_joint_start.assign(size_t(B) + 1, 0);
    for (int j = 0; j < J; ++j) {
        if (jparent[j] >= 0) h.body_joint_start[jparent[j] + 1]++;
        if (jchild[j] >= 0) h.body_joint_start[jchild[j] + 1]++;
    }
    for (int b = 0; b < B; ++b) h.body_joint_start[b + 1] += h.body_joint_start[b];
    h.body_joint_entry.assign(size_t(h.body_joint_start[B]), 0);
    {
        std::vector<int> fill(h.body_joint_start.begin(), h.body_joint_start.end() - 1);
        int e = 0;
        for (int j = 0; j < J; ++j) {
            while (e + 1 < E && j >= h.env_joint_start[e + 1]) ++e;
            int jl = j - h.env_joint_start[e];
            if (jparent[j] >= 0) h.body_joint_entry[fill[jparent[j]]++] = (jl << 1) | 0;
            if (jchild[j] >= 0) h.body_joint_entry[fill[jchild[j]]++] = (jl << 1) | 1;
            int bs = h.env_body_start[e], be = h.env_body_start[e + 1];
            if ((jparent[j] >= 0 && (jparent[j] < bs || jparent[j] >= be)) || jchild[j] < bs || jchild[j] >= be) {
                set_error("joint connects bodies of different worlds");
                return NB2_ERR_INVALID_ARGUMENT;
            }
        }
    }
    // ---- articulation tables for the Featherstone kernel ----------------------------------------
    {
        std::vector<int> janc, jqd, bflags, jtype, jdim;
        if ((st = fetch(d.joint_ancestor, size_t(J), janc))) return st;
        if ((st = fetch(d.joint_type, size_t(J), jtype))) return st;
        if ((st = fetch(d.joint_dof_dim, size_t(J) * 2, jdim))) return st;
        if ((st = fetch(d.body_flags, size_t(B), bflags))) return st;
        for (int j = 0; j < J; ++j)
            if (jchild[j] != j) {  // the reference's spatial_mass indexes body_I_s by joint index (kernels.py:1476-1477)
                h.featherstone_supported = false;
                h.featherstone_reason = "joint j must drive body j (the reference mass matrix assumes body index == joint index)";
            }
        if ((st = fetch(d.joint_qd_start, size_t(J) + 1, jqd))) return st;
        h.joint_depth.assign(size_t(J), 0);
        h.joint_anc_mask.assign(size_t(J), 0ull);
        h.art_H_start.assign(size_t(d.articulation_count) + 1, 0);
        h.env_H_start.assign(size_t(E) + 1, 0);
        int max_depth = 0;
        for (int a = 0; a < d.articulation_count; ++a) {
            const int j0 = art_start[a], j1 = art_start[a + 1];
            if (j1 - j0 > 64) {
                h.featherstone_supported = false;
                h.featherstone_reason = "articulations with more than 64 joints";
            }
            for (int j = j0; j < j1; ++j) {
                int anc = janc[j];
                if (anc >= j || (anc >= 0 && anc < j0)) {
                    h.featherstone_supported = false;
                    h.featherstone_reason = "joints must be stored parent-before-child inside their articulation";
                    h.fk_levels = false;  // eval_fk then walks the joints serially, in array order, like the reference
                    anc = -1;
                }
                h.joint_depth[j] = anc >= 0 ? h.joint_depth[anc] + 1 : 0;
                h.joint_anc_mask[j] = (anc >= 0 ? h.joint_anc_mask[anc] : 0ull) | (1ull << ((j - j0) & 63));
                max_depth = std::max(max_depth, h.joint_depth[j]);
                if (jart[j] != a) {
                    h.featherstone_supported = false;
                    h.featherstone_reason = "joints outside an articulation";
                }
            }
        }
        // ---- H-stage schedule (see DevModel): the per-(depth, dof number) column batches of every articulation ----------------
        h.joint_desc_mask.assign(size_t(J), 0ull);
        h.dof_joint.assign(size_t(jqd[J]), 0);
        h.art_batch_count.assign(size_t(d.articulation_count), 0);
        h.art_hb_body_start.assign(size_t(d.articulation_count), 0);
        h.art_hb_row_start.assign(size_t(d.articulation_count), 0);
        h.hb_body_col.clear();
        h.hb_row_col.clear();
        for (int a = 0; a < d.articulation_count && h.featherstone_supported; ++a) {
            const int j0 = art_start[a], j1 = art_start[a + 1], anj = j1 - j0;
            const int ad0 = jqd[j0], n = jqd[j1] - ad0;
            h.max_art_dofs = std::max(h.max_art_dofs, n);
            if (n > 127) {
                h.featherstone_supported = false;
                h.featherstone_reason = "articulations with more than 127 dofs";
                break;
            }
            int maxdep = 0;
            for (int j = j0; j < j1; ++j) {
                maxdep = std::max(maxdep, h.joint_depth[j]);
                for (int k = jqd[j]; k < jqd[j + 1]; ++k) h.dof_joint[k] = (signed char)(j - j0);
                unsigned long long m = 0ull;  // descendant-or-self: every joint i whose ancestor mask contains j
                for (int i = j0; i < j1; ++i) m |= ((h.joint_anc_mask[i] >> (j - j0)) & 1ull) << (i - j0);
                h.joint_desc_mask[j] = m;
            }
            // ancestor-or-self of joint i at a given depth (-1: i is shallower)
            auto anc_at = [&](int i, int dep) {
                int jb = -1;
                for (unsigned long long m = h.joint_anc_mask[j0 + i]; m; m &= m - 1ull) {
                    const int b = __builtin_ctzll(m);
                    if (h.joint_depth[j0 + b] == dep) jb = b;
                }
                return jb;
            };
            h.art_hb_body_start[a] = int(h.hb_body_col.size());
            h.art_hb_row_start[a] = int(h.hb_row_col.size());
            int batches = 0;
            for (int dep = 0; dep <= maxdep; ++dep)
                for (int kk = 0; kk < 6; ++kk) {
                    bool any = false;
                    for (int j = j0; j < j1 && !any; ++j) any = h.joint_depth[j] == dep && jqd[j + 1] - jqd[j] > kk;
                    if (!any) break;  // dof counts only shrink the batch
                    for (int i = 0; i < anj; ++i) {
                        const int jb = h.joint_depth[j0 + i] >= dep ? anc_at(i, dep) : -1;
                        const bool on = jb >= 0 && jqd[j0 + jb + 1] - jqd[j0 + jb] > kk;
                        h.hb_body_col.push_back(on ? (signed char)(jqd[j0 + jb] - ad0 + kk) : (signed char)-1);
                    }
                    for (int ra = 0; ra < n; ++ra) {
                        const int ja = h.dof_joint[ad0 + ra];
                        const int jb = h.joint_depth[j0 + ja] >= dep ? anc_at(ja, dep) : -1;
                        int col = -1;
                        if (jb >= 0 && jqd[j0 + jb + 1] - jqd[j0 + jb] > kk) col = jqd[j0 + jb] - ad0 + kk;
                        if (col > ra) col = -1;  // upper triangle (only possible inside joint(col) itself)
                        h.hb_row_col.push_back((signed char)col);
                    }
                    batches += 1;
                }
            h.art_batch_count[a] = batches;
        }
        {  // a body driven by two joints ("undefined semantics" upstream): only the serial walk reproduces the array-order result
            std::vector<char> driven(size_t(B), 0);
            for (int j = 0; j < J; ++j)
                if (jart[j] >= 0 && jchild[j] >= 0) {
                    if (driven[jchild[j]]) h.fk_levels = false;
                    driven[jchild[j]] = 1;
                }
        }
        int e = 0, max_env_H = 0, max_env_arts = 0;
        for (int ee = 0; ee < E; ++ee) {
            int acc = 0;
            for (int a = h.env_art_start[ee]; a < h.env_art_start[ee + 1]; ++a) {
                h.art_H_start[a] = acc;
                int nd = jqd[art_start[a + 1]] - jqd[art_start[a]];
                acc += nd * nd;
            }
            h.env_H_start[ee + 1] = h.env_H_start[ee] + acc;
            max_env_H = std::max(max_env_H, acc);
            max_env_arts = std::max(max_env_arts, h.env_art_start[ee + 1] - h.env_art_start[ee]);
        }
        (void)e;
        m->dev.max_depth = max_depth;
        m->dev.max_env_H = max_env_H;
        m->dev.max_env_arts = max_env_arts;
        int max_dofs = 0, max_coords = 0;
        std::vector<int> jq;
        if ((st = fetch(d.joint_q_start, size_t(J) + 1, jq))) return st;
        for (int ee = 0; ee < E; ++ee) {
            int ja = h.env_joint_start[ee], jb = h.env_joint_start[ee + 1];
            max_dofs = std::max(max_dofs, jqd[jb] - jqd[ja]);
            max_coords = std::max(max_coords, jq[jb] - jq[ja]);
        }
        m->dev.max_env_dofs = max_dofs;
        m->dev.max_env_coords = max_coords;
    }
    DevModel& dv = m->dev;
    dv.d = d;
    dv.env_count = E;
    dv.global_shape_count = int(h.global_shapes.size());
    dv.max_env_bodies = dv.max_env_joints = dv.max_env_slots_shapes = dv.max_env_pairs = dv.max_env_contact_slots = 0;
    for (int e = 0; e < E; ++e) {
        dv.max_env_bodies = std::max(dv.max_env_bodies, h.env_body_start[e + 1] - h.env_body_start[e]);
        dv.max_env_joints = std::max(dv.max_env_joints, h.env_joint_start[e + 1] - h.env_joint_start[e]);
        dv.max_env_slots_shapes =
            std::max(dv.max_env_slots_shapes, h.env_shape_start[e + 1] - h.env_shape_start[e] + dv.global_shape_count);
        dv.max_env_pairs = std::max(dv.max_env_pairs, h.env_pair_start[e + 1] - h.env_pair_start[e]);
        dv.max_env_contact_slots = std::max(dv.max_env_contact_slots, h.env_slot_start[e + 1] - h.env_slot_start[e]);
    }
    dv.slot_total = h.env_slot_start[E];
    dv.has_mesh_pairs = m->has_mesh_pairs ? 1 : 0;
    m->lanes_per_env =
        std::min(32, std::max(8, pow2_at_least(std::max({dv.max_env_bodies, dv.max_env_joints, std::min(dv.max_env_pairs, 32)}))));
    // small batches cannot fill the GPU with warps: give each environment a full warp so its contact / pair loops need fewer
    // rounds (measured on 512 box stacks: xpbd_step 90 -> 68 us); large batches keep the narrowest group that fits
    while (m->lanes_per_env < 32 && (long long)E * m->lanes_per_env / 32 < 4LL * m->sm_count) m->lanes_per_env *= 2;
    return NB2_OK;
}

static void free_allocations(nb2_model* m) {
    for (void* p : m->allocations) cudaFree(p);
    m->allocations.clear();
}

static nb2_status upload_tables(nb2_model* m) {
    HostTables& h = m->host;
    DevModel& dv = m->dev;
    nb2_status st;
    if ((st = upload(m, h.env_body_start, &dv.env_body_start))) return st;
    if ((st = upload(m, h.env_joint_start, &dv.env_joint_start))) return st;
    if ((st = upload(m, h.env_shape_start, &dv.env_shape_start))) return st;
    if ((st = upload(m, h.env_pair_start, &dv.env_pair_start))) return st;
    if ((st = upload(m, h.env_slot_start, &dv.env_slot_start))) return st;
    if ((st = upload(m, h.env_art_start, &dv.env_art_start))) return st;
    if ((st = upload(m, h.global_shapes, &dv.global_shapes))) return st;
    if ((st = upload(m, h.pairs, &dv.pairs))) return st;
    if ((st = upload(m, h.body_joint_start, &dv.body_joint_start))) return st;
    if ((st = upload(m, h.body_joint_entry, &dv.body_joint_entry))) return st;
    if ((st = upload(m, h.joint_depth, &dv.joint_depth))) return st;
    if ((st = upload(m, h.joint_anc_mask, &dv.joint_anc_mask))) return st;
    if ((st = upload(m, h.art_H_start, &dv.art_H_start))) return st;
    if ((st = upload(m, h.env_H_start, &dv.env_H_start))) return st;
    if ((st = upload(m, h.art_batch_count, &dv.art_batch_count))) return st;
    if ((st = upload(m, h.art_hb_body_start, &dv.art_hb_body_start))) return st;
    if ((st = upload(m, h.art_hb_row_start, &dv.art_hb_row_start))) return st;
    if ((st = upload(m, h.hb_body_col, &dv.hb_body_col))) return st;
    if ((st = upload(m, h.hb_row_col, &dv.hb_row_col))) return st;
    if ((st = upload(m, h.joint_desc_mask, &dv.joint_desc_mask))) return st;
    if ((st = upload(m, h.dof_joint, &dv.dof_joint))) return st;
    void* p = nullptr;
    {
        size_t nL = std::max<size_t>(size_t(h.env_H_start.back()), 1);
        NB2_CUDA_CHECK(cudaMalloc(&p, nL * sizeof(float)));
        NB2_CUDA_CHECK(cudaMemset(p, 0, nL * sizeof(float)));
        m->allocations.push_back(p);
        dv.fs_L = static_cast<float*>(p);
    }
    {
        size_t n = std::max<size_t>(size_t(dv.slot_total) * 6, 1) * sizeof(float);
        NB2_CUDA_CHECK(cudaMalloc(&p, n));
        NB2_CUDA_CHECK(cudaMemset(p, 0, n));
        m->allocations.push_back(p);
        dv.contact_impulse = static_cast<float*>(p);
        n = std::max<size_t>(size_t(dv.d.joint_count) * 6, 1) * sizeof(float);
        NB2_CUDA_CHECK(cudaMalloc(&p, n));
        NB2_CUDA_CHECK(cudaMemset(p, 0, n));
        m->allocations.push_back(p);
        dv.joint_impulse = static_cast<float*>(p);
    }
    size_t cb_bytes = std::max<size_t>(size_t(dv.slot_total) * CF_COUNT, 1) * sizeof(float);
    NB2_CUDA_CHECK(cudaMalloc(&p, cb_bytes));
    NB2_CUDA_CHECK(cudaMemset(p, 0, cb_bytes));
    m->allocations.push_back(p);
    dv.cb = static_cast<float*>(p);
    NB2_CUDA_CHECK(cudaMalloc(&p, (size_t(dv.env_count) + 1) * sizeof(int)));
    NB2_CUDA_CHECK(cudaMemset(p, 0, (size_t(dv.env_count) + 1) * sizeof(int)));
    m->allocations.push_back(p);
    dv.env_contact_count = static_cast<int*>(p);
    NB2_CUDA_CHECK(cudaMalloc(&p, (size_t(dv.env_count) + 1) * sizeof(int)));
    NB2_CUDA_CHECK(cudaMemset(p, 0, (size_t(dv.env_count) + 1) * sizeof(int)));
    m->allocations.push_back(p);
    dv.env_contact_offset = static_cast<int*>(p);
    return NB2_OK;
}


// Frees one tracked device allocation (the contact blocks are re-sized when the broad phase changes).
static void release(nb2_model* m, const void* p) {
    if (!p) return;
    for (size_t i = 0; i < m->allocations.size(); ++i)
        if (m->allocations[i] == p) {
            cudaFree(m->allocations[i]);
            m->allocations.erase(m->allocations.begin() + i);
            return;
        }
}

// Contact-block slot ranges + buffers for the current pair source: 5 slots per explicit pair, or per candidate-capacity pair of
// the run-time broad phases.
static nb2_status allocate_contact_blocks(nb2_model* m) {
    DevModel& dv = m->dev;
    HostTables& h = m->host;
    const int E = dv.env_count;
    release(m, dv.env_slot_start);
    release(m, dv.cb);
    release(m, dv.contact_impulse);
    dv.max_env_contact_slots = 0;
    for (int e = 0; e < E; ++e) dv.max_env_contact_slots = std::max(dv.max_env_contact_slots, h.env_slot_start[e + 1] - h.env_slot_start[e]);
    dv.slot_total = h.env_slot_start[E];
    nb2_status st;
    if ((st = upload(m, h.env_slot_start, &dv.env_slot_start))) return st;
    void* p = nullptr;
    size_t n = std::max<size_t>(size_t(dv.slot_total) * 6, 1) * sizeof(float);
    NB2_CUDA_CHECK(cudaMalloc(&p, n));
    NB2_CUDA_CHECK(cudaMemset(p, 0, n));
    m->allocations.push_back(p);
    dv.contact_impulse = static_cast<float*>(p);
    n = std::max<size_t>(size_t(dv.slot_total) * CF_COUNT, 1) * sizeof(float);
    NB2_CUDA_CHECK(cudaMalloc(&p, n));
    NB2_CUDA_CHECK(cudaMemset(p, 0, n));
    m->allocations.push_back(p);
    dv.cb = static_cast<float*>(p);
    NB2_CUDA_CHECK(cudaMemset(dv.env_contact_count, 0, (size_t(E) + 1) * sizeof(int)));
    return NB2_OK;
}

static nb2_status configure_broad_phase(nb2_model* m, int mode, int max_pairs, bool include_static_kinematic) {
    DevModel& dv = m->dev;
    HostTables& h = m->host;
    const int E = dv.env_count;
    dv.include_static_kinematic_pairs = include_static_kinematic ? 1 : 0;
    if (mode == dv.broad_phase && (mode == NB2_BROAD_PHASE_EXPLICIT || max_pairs == m->dyn_pairs_requested)) return NB2_OK;
    release(m, dv.dyn_pairs);
    release(m, dv.env_dyn_count);
    dv.dyn_pairs = nullptr;
    dv.env_dyn_count = nullptr;
    dv.dyn_pair_cap = 0;
    if (mode != NB2_BROAD_PHASE_EXPLICIT && m->has_mesh_pairs) {
        set_error("nb2_collide_configure: MESH shapes are supported with the explicit broad phase only");
        return NB2_ERR_UNSUPPORTED;
    }
    if (mode == NB2_BROAD_PHASE_EXPLICIT) {
        h.env_slot_start = h.explicit_env_slot_start;  // 5 per pair, one per vertex for mesh-plane pairs
        m->max_env_contacts = m->explicit_max_env_contacts;
        m->has_convex_pairs = m->explicit_has_convex_pairs;
    } else {
        if (dv.max_env_slots_shapes > 65535) {
            set_error("nb2_collide_configure: more than 65535 shapes in one world");
            return NB2_ERR_CAPACITY;
        }
        if (!dv.d.shape_collision_group) {
            set_error("nb2_collide_configure: broad_phase nxn / sap needs model.shape_collision_group");
            return NB2_ERR_INVALID_ARGUMENT;
        }
        int cap = 0;
        std::vector<int> caps(size_t(E), 0);
        for (int e = 0; e < E; ++e) {
            const long long ns = h.env_shape_start[e + 1] - h.env_shape_start[e] + dv.global_shape_count;
            long long c = ns * (ns - 1) / 2;
            if (max_pairs > 0) c = std::min<long long>(c, max_pairs);
            caps[e] = int(std::min<long long>(c, 1 << 20));
            cap = std::max(cap, caps[e]);
        }
        for (int e = 0; e < E; ++e) h.env_slot_start[e + 1] = h.env_slot_start[e] + 5 * caps[e];
        if (h.env_slot_start[E] < 0 || (long long)E * cap > (1ll << 30)) {
            set_error("nb2_collide_configure: candidate capacity too large; pass max_pairs_per_world (CollisionPipeline(shape_pairs_max=...))");
            return NB2_ERR_CAPACITY;
        }
        dv.dyn_pair_cap = cap;
        void* p = nullptr;
        NB2_CUDA_CHECK(cudaMalloc(&p, std::max<size_t>(size_t(E) * cap, 1) * sizeof(int2)));
        m->allocations.push_back(p);
        dv.dyn_pairs = static_cast<int2*>(p);
        NB2_CUDA_CHECK(cudaMalloc(&p, (size_t(E) + 1) * sizeof(int)));
        NB2_CUDA_CHECK(cudaMemset(p, 0, (size_t(E) + 1) * sizeof(int)));
        m->allocations.push_back(p);
        dv.env_dyn_count = static_cast<int*>(p);
        m->max_env_contacts = 5 * cap;
        m->has_convex_pairs = true;  // any type pair may show up at run time
        // excluded pairs -> sorted 64-bit keys
        release(m, dv.filter_keys);
        dv.filter_keys = nullptr;
        dv.filter_count = 0;
        if (dv.d.shape_collision_filter_pair_count > 0 && dv.d.shape_collision_filter_pairs) {
            std::vector<int> fp;
            nb2_status st = fetch(dv.d.shape_collision_filter_pairs, size_t(dv.d.shape_collision_filter_pair_count) * 2, fp);
            if (st != NB2_OK) return st;
            std::vector<long long> keys;
            keys.reserve(fp.size() / 2);
            for (size_t i = 0; i + 1 < fp.size(); i += 2) {
                const long long a = std::min(fp[i], fp[i + 1]), b = std::max(fp[i], fp[i + 1]);
                keys.push_back((a << 32) | b);
            }
            std::sort(keys.begin(), keys.end());
            keys.erase(std::unique(keys.begin(), keys.end()), keys.end());
            const long long* dk = nullptr;
            if ((st = upload(m, keys, &dk))) return st;
            dv.filter_keys = dk;
            dv.filter_count = int(keys.size());
        }
    }
    dv.broad_phase = mode;
    m->dyn_pairs_requested = max_pairs;
    return allocate_contact_blocks(m);
}

// Every entry point runs on the model's device and leaves the caller's current device as it found it (a process may drive
// several GPUs; nb2_model_destroy is called from a garbage collector at arbitrary points).
struct DeviceGuard {
    int prev = -1, dev = -1;
    explicit DeviceGuard(int device) : dev(device) {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != dev) cudaSetDevice(dev);
    }
    ~DeviceGuard() {
        if (prev >= 0 && prev != dev) cudaSetDevice(prev);
    }
};

}  // namespace nb2

using namespace nb2;

extern "C" {

nb2_status nb2_model_create(const nb2_model_desc* desc, int32_t device, nb2_model** out) {
    if (!desc || !out) {
        set_error("nb2_model_create: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    *out = nullptr;
    DeviceGuard guard(device);
    int sm_count = 0;
    NB2_CUDA_CHECK(cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, device));
    nb2_model* m = new nb2_model();
    m->device = device;
    m->sm_count = sm_count;
    nb2_status st = build_tables(m, *desc);
    if (st == NB2_OK) st = upload_tables(m);
    if (st != NB2_OK) {
        free_allocations(m);
        delete m;
        return st;
    }
    m->explicit_max_env_contacts = m->max_env_contacts;
    m->explicit_has_convex_pairs = m->has_convex_pairs;
    m->dev.include_static_kinematic_pairs = 1;
    *out = m;
    return NB2_OK;
}

void nb2_model_destroy(nb2_model* model) {
    if (!model) return;
    DeviceGuard guard(model->device);
    for (void* p : {(void*)model->match_new_keys, (void*)model->match_prev_keys, (void*)model->match_prev_claim, (void*)model->match_prev_pos,
                    (void*)model->match_prev_normal, (void*)model->match_prev_count, (void*)model->match_prev_record,
                    (void*)model->match_prev_was_matched})
        if (p) cudaFree(p);
    free_allocations(model);
    delete model;
}

nb2_status nb2_model_notify_changed(nb2_model* model, const nb2_model_desc* desc, int32_t flags) {
    (void)flags;
    if (!model || !desc) {
        set_error("nb2_model_notify_changed: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    // The kernels read the Model arrays live; only refresh the borrowed pointers (topology changes need a new model).
    const nb2_model_desc& o = model->dev.d;
    if (desc->body_count != o.body_count || desc->joint_count != o.joint_count || desc->shape_count != o.shape_count ||
        desc->shape_pair_count != o.shape_pair_count || desc->world_count != o.world_count ||
        desc->articulation_count != o.articulation_count || desc->joint_dof_count != o.joint_dof_count ||
        desc->joint_coord_count != o.joint_coord_count || desc->gravity_count != o.gravity_count) {
        set_error("nb2_model_notify_changed: topology changed; create a new nb2_model");
        return NB2_ERR_UNSUPPORTED;
    }
    model->dev.d = *desc;
    return NB2_OK;
}

int32_t nb2_model_rigid_contact_max(const nb2_model* model) { return model ? model->dev.slot_total : 0; }

nb2_status nb2_collide_configure(nb2_model* model, int32_t broad_phase, int32_t max_pairs_per_world, int32_t include_static_kinematic_pairs) {
    if (!model || broad_phase < NB2_BROAD_PHASE_EXPLICIT || broad_phase > NB2_BROAD_PHASE_SAP || max_pairs_per_world < 0) {
        set_error("nb2_collide_configure: invalid argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return configure_broad_phase(model, broad_phase, max_pairs_per_world, include_static_kinematic_pairs != 0);
}

nb2_status nb2_collide(nb2_model* model, const float* body_q, const nb2_contacts_view* contacts, void* cuda_stream) {
    if (!model || (!body_q && model->dev.d.body_count > 0)) {
        set_error("nb2_collide: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    model->dev.export_rank = nullptr;  // a fresh export is in (world, key) order until nb2_contacts_sort runs
    model->contacts_imported = false;
    model->dev.spec_mode = 0;
    model->dev.spec_body_qd = nullptr;
    model->dev.spec_dt = model->dev.spec_max_ext = 0.0f;
    DeviceGuard guard(model->device);
    return launch_collide(model, body_q, contacts, static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_collide_speculative(nb2_model* model, const float* body_q, const float* body_qd, float dt, float max_speculative_extension,
                                   const nb2_contacts_view* contacts, void* cuda_stream) {
    if (!model || ((!body_q || !body_qd) && model->dev.d.body_count > 0)) {
        set_error("nb2_collide_speculative: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (!(dt >= 0.0f) || !(max_speculative_extension >= 0.0f) || std::isinf(dt) || std::isinf(max_speculative_extension)) {
        set_error("nb2_collide_speculative: dt and max_speculative_extension must be non-negative finite numbers");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (!model->dev.d.shape_collision_aabb_lower || !model->dev.d.shape_collision_aabb_upper || !model->dev.d.body_com) {
        set_error("nb2_collide_speculative: model.shape_collision_aabb_lower / _upper / body_com are required");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    model->dev.export_rank = nullptr;
    model->contacts_imported = false;
    // speculative_active (sim/collide.py:1831): without a horizon or an extension only the writer's admission rule differs
    model->dev.spec_mode = (dt > 0.0f && max_speculative_extension > 0.0f) ? 2 : 1;
    model->dev.spec_body_qd = body_qd;
    model->dev.spec_dt = dt;
    model->dev.spec_max_ext = max_speculative_extension;
    DeviceGuard guard(model->device);
    const nb2_status st = launch_collide(model, body_q, contacts, static_cast<cudaStream_t>(cuda_stream));
    model->dev.spec_mode = 0;
    model->dev.spec_body_qd = nullptr;
    return st;
}

nb2_status nb2_contacts_sort(nb2_model* model, const nb2_contacts_view* c, void* cuda_stream) {
    if (!model || !c || !c->rigid_contact_count || !c->shape0 || !c->shape1 || !c->point0 || !c->point1 || !c->offset0 || !c->offset1 ||
        !c->normal || !c->margin0 || !c->margin1 || c->rigid_contact_max < 0) {
        set_error("nb2_contacts_sort: NULL argument / contacts view has NULL arrays");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return launch_contacts_sort(model, *c, static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_contacts_import(nb2_model* model, const nb2_contacts_view* c, void* cuda_stream) {
    if (!model || !c || !c->rigid_contact_count || !c->shape0 || !c->shape1 || !c->point0 || !c->point1 || !c->offset0 || !c->offset1 ||
        !c->normal || !c->margin0 || !c->margin1 || c->rigid_contact_max < 0) {
        set_error("nb2_contacts_import: NULL argument / contacts view has NULL arrays");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    model->contacts_imported = true;
    return launch_contacts_import(model, *c, static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_xpbd_step(nb2_model* model, const nb2_xpbd_params* params, const nb2_state_view* state_in,
                         const nb2_state_view* state_out, const nb2_control_view* control, int32_t use_contacts, float dt,
                         void* cuda_stream) {
    if (!model || !params || !state_in || !state_out || !control) {
        set_error("nb2_xpbd_step: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (params->iterations < 0 || !(dt > 0.0f)) {
        set_error("nb2_xpbd_step: iterations must be >= 0 and dt > 0");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if ((use_contacts & NB2_XPBD_CONTACT_IMPULSE) && (use_contacts & NB2_XPBD_USE_CONTACTS)) model->xpbd_impulse_dt = dt;
    DeviceGuard guard(model->device);
    return launch_xpbd_step(model, *params, *state_in, *state_out, *control, use_contacts, dt,
                            static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_xpbd_update_contacts(nb2_model* model, const nb2_contacts_view* contacts, void* cuda_stream) {
    if (!model || !contacts || !contacts->force || !contacts->rigid_contact_count) {
        set_error("nb2_xpbd_update_contacts: NULL argument (contacts.force must be allocated)");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (!(model->xpbd_impulse_dt > 0.0f)) {
        set_error("nb2_xpbd_update_contacts: no contact impulse data available, run nb2_xpbd_step with NB2_XPBD_CONTACT_IMPULSE first");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return launch_xpbd_update_contacts(model, *contacts, static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_integrate_bodies(nb2_model* model, const nb2_state_view* state_in, const nb2_state_view* state_out,
                                float angular_damping, float dt, void* cuda_stream) {
    if (!model || !state_in || !state_out) {
        set_error("nb2_integrate_bodies: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return launch_integrate_bodies(model, *state_in, *state_out, angular_damping, dt, static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_featherstone_step(nb2_model* model, const nb2_featherstone_params* params, const nb2_state_view* state_in,
                                 const nb2_state_view* state_out, const nb2_control_view* control, int32_t use_contacts,
                                 float dt, void* cuda_stream) {
    if (!model || !params || !state_in || !state_out || !control) {
        set_error("nb2_featherstone_step: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return launch_featherstone_step(model, *params, *state_in, *state_out, *control, use_contacts, dt,
                                    static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_eval_fk(nb2_model* model, const float* joint_q, const float* joint_qd, float* body_q, float* body_qd,
                       void* cuda_stream) {
    if (!model || !joint_q || !joint_qd || !body_q || !body_qd) {
        set_error("nb2_eval_fk: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return launch_eval_fk(model, joint_q, joint_qd, body_q, body_qd, static_cast<cudaStream_t>(cuda_stream));
}

nb2_status nb2_eval_fk_masked(nb2_model* model, const float* joint_q, const float* joint_qd, float* body_q, float* body_qd,
                              const uint8_t* articulation_mask, const int32_t* articulation_indices, int32_t index_count,
                              int32_t body_flag_filter, void* cuda_stream) {
    if (!model || !joint_q || !joint_qd || !body_q || !body_qd) {
        set_error("nb2_eval_fk_masked: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (articulation_mask && articulation_indices) {
        set_error("nb2_eval_fk_masked: cannot specify both mask and indices");  // sim/articulation.py:529-530
        return NB2_ERR_INVALID_ARGUMENT;
    }
    if (articulation_indices && index_count < 0) {
        set_error("nb2_eval_fk_masked: negative index_count");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return launch_eval_fk(model, joint_q, joint_qd, body_q, body_qd, static_cast<cudaStream_t>(cuda_stream), articulation_mask,
                          articulation_indices, index_count, body_flag_filter);
}

nb2_status nb2_eval_ik(nb2_model* model, const float* body_q, const float* body_qd, float* joint_q, float* joint_qd,
                       void* cuda_stream) {
    if (!model || !body_q || !body_qd || !joint_q || !joint_qd) {
        set_error("nb2_eval_ik: NULL argument");
        return NB2_ERR_INVALID_ARGUMENT;
    }
    DeviceGuard guard(model->device);
    return launch_eval_ik(model, body_q, body_qd, joint_q, joint_qd, static_cast<cudaStream_t>(cuda_stream));
}

const char* nb2_last_error(void) { return g_last_error.c_str(); }
int64_t nb2_kernel_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }
const char* nb2_version(void) { return "newton_b200 0.1 (sm_100a)"; }

}  // extern "C"
