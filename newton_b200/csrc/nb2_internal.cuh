// nb2_internal.cuh - private definitions shared by the translation units of libnewton_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/newton_b200.h"

namespace nb2 {

// Number of float/int fields of one contact slot in the env-major contact blocks (DESIGN.md "contact hand-off").
// Field f of slot s lives at cb[f * slot_total + s]: lanes read consecutive slots -> coalesced 128-byte lines.
enum ContactField {
    CF_BODY_A = 0,  // int: env-local body index or -1
    CF_BODY_B,
    CF_SHAPE0,  // int: model shape ids (for export)
    CF_SHAPE1,
    CF_P0X, CF_P0Y, CF_P0Z,     // point0 (body frame of A)
    CF_P1X, CF_P1Y, CF_P1Z,     // point1 (body frame of B)
    CF_O0X, CF_O0Y, CF_O0Z,     // offset0
    CF_O1X, CF_O1Y, CF_O1Z,     // offset1
    CF_NX, CF_NY, CF_NZ,        // normal A->B (world)
    CF_MARGIN0, CF_MARGIN1,
    CF_MU, CF_MU_TORSIONAL, CF_MU_ROLLING,  // pair-averaged friction coefficients
    CF_KE, CF_KD, CF_KF, CF_KA,             // pair-averaged penalty parameters (Featherstone / semi-implicit contact)
    CF_COUNT
};

// Everything a kernel needs, passed by value (all pointers are device pointers).
struct DevModel {
    nb2_model_desc d;           // the reference-layout Model arrays (borrowed)
    int env_count;
    const int* env_body_start;     // [E+1]
    const int* env_joint_start;    // [E+1]
    const int* env_shape_start;    // [E+1] env-local shapes
    const int* env_pair_start;     // [E+1] into pairs[]
    const int* env_slot_start;     // [E+1] contact-block slot ranges
    const int* env_art_start;      // [E+1] articulations
    const int* global_shapes;      // ids of world -1 shapes, appended to every env's slot table
    int global_shape_count;
    const int2* pairs;             // per env: (slot_a, slot_b), type-ordered (type_a <= type_b), sorted by contact key
    const int* body_joint_start;   // [B+1] CSR of (joint_local << 1 | is_child) in joint order
    const int* body_joint_entry;
    float* cb;                     // contact blocks: CF_COUNT planes of slot_total words
    int slot_total;
    int* env_contact_count;        // [E]
    int* env_contact_offset;       // [E+1] exclusive scan, written by the export path
    int max_env_bodies, max_env_joints, max_env_slots_shapes, max_env_pairs, max_env_contact_slots;
    // articulated-body (Featherstone) tables
    const int* joint_depth;            // [J] depth of each joint in its articulation tree (root = 0)
    const unsigned long long* joint_anc_mask;  // [J] bit k set <=> articulation-local joint k is an ancestor-or-self
    const int* art_H_start;            // [A+1] offset of each articulation's nd x nd block inside its env's H storage
    const int* env_H_start;            // [E+1] global offset of the env's H/L storage (persistent L for update intervals)
    float* fs_L;                       // persistent Cholesky factors [env_H_start[E]]
    int max_depth, max_env_dofs, max_env_coords, max_env_H, max_env_arts;
    // H = J^T M J schedule, derived from the joint tree at nb2_model_create (the kernel indexes, it does not walk bit masks):
    // columns of H are formed in batches of (tree depth, dof number inside the joint) - joints of one batch are never ancestors of
    // one another, so every body and every row sees at most one column per batch
    const int* art_batch_count;        // [A]   batches of the articulation
    const int* art_hb_body_start;      // [A]   offset into hb_body_col: batch-major, anj entries per batch
    const int* art_hb_row_start;       // [A]   offset into hb_row_col: batch-major, n (dofs) entries per batch
    const signed char* hb_body_col;    // articulation-local dof (column) whose P_i = I_i S_col body i forms in this batch, or -1
    const signed char* hb_row_col;     // column whose entry H[row, col] row `row` sums in this batch (col <= row), or -1
    const unsigned long long* joint_desc_mask;  // [J] bit i set <=> articulation-local body i hangs below (or is driven by) joint j
    const signed char* dof_joint;      // [D] articulation-local joint owning each dof
    // XPBD reporting scratch (row a17): weighted contact impulses (6 planes of slot_total) and per-joint child-side impulses
    float* contact_impulse;
    float* joint_impulse;  // [6 * joint_count]
    // exported index -> position after nb2_contacts_sort (nullptr: export order is the final order)
    const int* export_rank;
    // run-time broad phase (nb2_collide_configure): candidates of env e are dyn_pairs[e * dyn_pair_cap ...), env_dyn_count[e] of them
    // (may exceed the capacity: the excess was dropped), in the (slot_a, slot_b) type-ordered, key-sorted format of `pairs`
    int broad_phase;                 // NB2_BROAD_PHASE_*
    int include_static_kinematic_pairs;
    int dyn_pair_cap;
    int2* dyn_pairs;
    int* env_dyn_count;
    const long long* filter_keys;    // excluded pairs as (min << 32 | max), ascending
    int filter_count;
    // speculative contacts (nb2_collide_speculative): 0 = off, 1 = enabled but inactive for this call (dt == 0 or extension == 0:
    // only the writer's admission rule changes), 2 = active (shape velocities, swept broad phase, velocity-extended search gaps)
    int spec_mode;
    int has_mesh_pairs;    // the explicit pair list holds (mesh, infinite plane) pairs
    const float* spec_body_qd;
    float spec_dt, spec_max_ext;
};

// explicit pair list: bit set on .y of a (mesh slot, plane slot) pair - one contact per mesh vertex (narrow_phase.py:1761-1861)
enum : int { NB2_PAIR_MESH_PLANE = 0x40000000 };

struct HostTables {
    std::vector<int> env_body_start, env_joint_start, env_shape_start, env_pair_start, env_slot_start, env_art_start;
    std::vector<int> explicit_env_slot_start;  // slot ranges of the explicit pair list (restored when the broad phase goes back to it)
    std::vector<int> global_shapes;
    std::vector<int2> pairs;
    std::vector<int> body_joint_start, body_joint_entry;
    std::vector<int> joint_depth, art_H_start, env_H_start;
    std::vector<unsigned long long> joint_anc_mask, joint_desc_mask;
    std::vector<int> art_batch_count, art_hb_body_start, art_hb_row_start;
    std::vector<signed char> hb_body_col, hb_row_col, dof_joint;
    int max_art_dofs = 0;  // largest articulation (dofs)
    bool featherstone_supported = true;
    bool fk_levels = true;     // eval_fk may schedule joints by tree depth (parent-before-child order, one driving joint per body)
    std::string featherstone_reason;
};

}  // namespace nb2

struct nb2_model {
    int device = 0;
    int sm_count = 0;        // multiprocessors of `device`, queried at nb2_model_create
    nb2::DevModel dev{};
    nb2::HostTables host;
    std::vector<void*> allocations;
    int lanes_per_env = 32;  // sub-warp group width used by the fused kernels
    int featherstone_step_count = 0;
    // scratch of nb2_contacts_import (allocated on first use, sized by the imported buffer's capacity)
    int import_capacity = 0;
    int *import_keys = nullptr, *import_keys_sorted = nullptr, *import_idx = nullptr, *import_idx_sorted = nullptr;
    void* import_temp = nullptr;
    size_t import_temp_bytes = 0;
    // scratch of nb2_contacts_sort (deterministic=True export order)
    int sort_capacity = 0;
    unsigned long long *sort_keys = nullptr, *sort_keys_sorted = nullptr;
    int *sort_idx = nullptr, *sort_idx_sorted = nullptr;
    float* sort_stage = nullptr;  // 20 words per contact: a copy of the exported arrays to gather from
    int* sort_rank = nullptr;     // exported index -> sorted position
    void* sort_temp = nullptr;
    size_t sort_temp_bytes = 0;
    // contact matching history (nb2_contacts_match): previous frame's sorted keys / world midpoints / normals / claim words
    int match_capacity = 0;
    long long *match_new_keys = nullptr, *match_prev_keys = nullptr, *match_prev_claim = nullptr;
    float *match_prev_pos = nullptr, *match_prev_normal = nullptr;
    int* match_prev_count = nullptr;
    float* match_prev_record = nullptr;      // sticky: [4][capacity] vec3 - point0, point1, offset0, offset1 of the saved frame
    int* match_prev_was_matched = nullptr;   // contact_report: 1 where a contact of this frame kept the saved row
    bool match_prev_has_record = false;      // the saved frame carries sticky records (the last save ran in sticky mode)
    bool implicit_single = false;  // model built without begin_world(): one environment holding every entity
    bool has_convex_pairs = false;  // some pair's types have no analytic collider -> collide_kernel<L, true>
    bool has_mesh_pairs = false;    // the explicit pair list holds (mesh, infinite plane) pairs (flag NB2_PAIR_MESH_PLANE on .y)
    int explicit_max_env_contacts = 0, dyn_pairs_requested = 0;
    bool explicit_has_convex_pairs = false;
    int max_env_contacts = 0;       // max over envs of the sum of the pairs' own contact maxima (<= 4 analytic, <= 5 manifold)
    bool contacts_imported = false; // the contact blocks hold an imported foreign buffer (any count up to the slot range)
    float xpbd_impulse_dt = 0.0f;  // dt of the last nb2_xpbd_step that accumulated contact impulses (0 = none yet)
};

namespace nb2 {
// Warps per SM a launch with one environment per L-lane group needs to cover the batch in one wave.  The fused kernels' launchers
// pick their CTA width from it.
inline long long warps_per_sm(const nb2_model* m, int L) {
    const long long total_warps = (m->dev.env_count + (32 / L) - 1) / (32 / L);
    return (total_warps + m->sm_count - 1) / m->sm_count;
}
void set_error(const std::string& msg);
void count_launch(int n = 1);
nb2_status launch_collide(nb2_model* m, const float* body_q, const nb2_contacts_view* contacts, cudaStream_t s);
nb2_status launch_broadphase(nb2_model* m, const float* body_q, cudaStream_t s);
nb2_status launch_xpbd_step(nb2_model* m, const nb2_xpbd_params& p, const nb2_state_view& in, const nb2_state_view& out,
                            const nb2_control_view& ctl, int use_contacts, float dt, cudaStream_t s);
nb2_status launch_contacts_sort(nb2_model* m, const nb2_contacts_view& contacts, cudaStream_t s);
nb2_status launch_contacts_import(nb2_model* m, const nb2_contacts_view& contacts, cudaStream_t s);
nb2_status launch_xpbd_update_contacts(nb2_model* m, const nb2_contacts_view& contacts, cudaStream_t s);
nb2_status launch_integrate_bodies(nb2_model* m, const nb2_state_view& in, const nb2_state_view& out, float angular_damping,
                                   float dt, cudaStream_t s);
nb2_status launch_featherstone_step(nb2_model* m, const nb2_featherstone_params& p, const nb2_state_view& in,
                                    const nb2_state_view& out, const nb2_control_view& ctl, int use_contacts, float dt,
                                    cudaStream_t s);
nb2_status launch_eval_fk(nb2_model* m, const float* joint_q, const float* joint_qd, float* body_q, float* body_qd,
                          cudaStream_t s, const uint8_t* mask = nullptr, const int* indices = nullptr, int index_count = 0,
                          int body_flag_filter = 3);
nb2_status launch_eval_ik(nb2_model* m, const float* body_q, const float* body_qd, float* joint_q, float* joint_qd, cudaStream_t s);
}  // namespace nb2

#define NB2_CUDA_CHECK(expr)                                                                          \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess) {                                                                      \
            nb2::set_error(std::string(#expr) + ": " + cudaGetErrorString(_e));                       \
            return NB2_ERR_CUDA;                                                                      \
        }                                                                                             \
    } while (0)
