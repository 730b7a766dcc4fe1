// Device-side data model of the batched Real3D-Aug engine (one instance per GPU / process).
//
// HBM layout (B = scans in the batch, P = max_points + max_inserted, K = yaw_steps, HW = rows * cols):
//   xyzi      float4 [B][max_points]   original points exactly as read from velodyne/*.bin (immutable)
//   tail_*    double [B][max_inserted] inserted object points keep their fp64 coordinates (the reference keeps the
//                                       working cloud in float64 until save_data casts, od/ds:86-88)
//   label     u32    [B][P]            semantic label (original) / object label (inserted)
//   r, el     double [B][P]            cached range / elevation (A2 is computed ONCE per point, not once per slot)
//   col       u16    [B][P]            cached azimuth bin (depends only on the image width)
//   pix       i32    [B][P]            pix_id of the current slot's projection
//   alive     u8     [B][P]            0 once an occlusion removed the point (scene = scene[keep] in the reference)
//   zraw      u64    [B][HW]           z-buffer: min range bits per pixel, all-ones = empty
//   smooth    double [B][HW]           range image after closing + hole fill (500 = empty)
//   obj_raw   u64    [B][HW]           scratch z-buffer of the chosen candidate (kept all-ones between uses)
//   dmask     u32    [B][HW/32]        vis_px bit mask of the last evaluated candidate (od/ins:486)
//   cand_*           [B][K+1]          per-candidate results of the current try (index = rotation 1..K)
#pragma once
#include "r3d_common.cuh"
#include "../../include/real3d_b200.h"

namespace r3d {

enum : int { PH_INIT = 0, PH_AFTER_TRY = 1, PH_DONE = 2, PH_ERROR = 3 };
enum : unsigned { CF_ONMAP = 1u, CF_HOK = 2u };
constexpr int APT_IDX_BITS = 27;                       // apts.w = (surface slot << 27) | point index
constexpr unsigned APT_IDX_MASK = (1u << APT_IDX_BITS) - 1u, APT_SLOT_NONE = 15u;

struct ClassCfg {
    int min_points, map_sel;
    unsigned map_ok_mask;
    int pedestrian, n_surface;
    int surface[R3D_MAX_SURFACE];
    unsigned ok_slots;   // bit i: EngineDev::surf_all[i] is one of this class's surface labels
};

struct ObjBox {          // one cut object: box from read_label_line (od/fs:175-224, ss/fs:155-189), host-prepared
    double cx, cy, cz;   // cz = box bottom
    double a, b;         // R0[0][0], R0[1][0]
    double length, width, height;
    double rho, psi0;    // range / azimuth of the box centre about the sensor (pruning only)
    double reach;        // horizontal bounding radius (pruning only)
    // extent of the object's POINTS in the box frame (they may stick out of the annotated box: the cut-out box of
    // object_cut_out.py:133 is 5 cm wider per side than the box read_label_line parses): along the box x / y axis
    // relative to the box centre and in z relative to the box bottom, padded by 1e-6 m.  Invariant under the candidate
    // rotations (points and box turn together); used only to prune the object-points-vs-scene-box test.
    double eu0, eu1, ev0, ev1, ez0, ez1;
    int cls, first, count, pad;
};

struct ScanState {
    int n0, n_tail, tail_before, n_boxes;
    int phase, status;
    int remaining[R3D_MAX_CLASSES];
    int inserted_class, timeout, start_idx, end_idx, s_idx, event;
    int cur_class, cur_obj;
    int try_active, need_project, apply_flag, dirty, scene_changed;
    int n_feasible, found_rank, chosen_rot, accepted, chosen_v;
    int n_inserted, n_check;
    int far_flag;
    int first, extreme_removed;          // first slot of the scan / a removed point held the min or max elevation
    int d_r0, d_r1, d_c0, d_c1;          // pixel rectangle (inclusive) that contains every bit of dmask
    unsigned long long new_min_bits, new_max_bits;   // elevation range of the points the last accept appended
    int win_x0, win_y0;
    unsigned long long min_el_bits, max_el_bits;
    ImageGeom geom;
    long long walk_cycles;               // SM cycles the scan's walker CTA lived in the last run (diagnostics)
    int walk_tries, walk_pad;
};

struct EngineDev {       // passed by value to kernels
    int task, rows, cols, hw, K, max_tries, n_classes;
    int B, max_points, max_inserted, P, max_boxes, max_events, max_obj_points;
    int road_label, n_road_indexes, map_window, dwords, n_objects, n_perm_events;
    int road_indexes[R3D_MAX_SURFACE];
    // semseg: the distinct labels some class may stand on (ss/fs:92-93).  Entries of the all-points grid carry the slot of
    // their label (APT_SLOT_NONE = none of them) above the point index, so the collision test drops the ground points
    // a class accepts before any arithmetic
    int n_surf_all, surf_all[15];
    double step_rad;
    int G;                            // road-level grid side in cells
    float grid_inv_cell;
    double grid_cell;
    int* gcell;                       // [B][G*G]   CSR end offsets (cell c holds gpts[gcell[c-1] .. gcell[c]) )
    float4* gpts;                     // [B][max_points]  surface points sorted by cell: x, y, z, label bits
    unsigned char* gnear;             // [B][G*G]   Chebyshev distance (cells, capped) to the nearest non-empty cell of gcell
    unsigned char* gscratch;          // [B][G*G]   row pass of the distance transform
    int* acell;                       // [B][G*G]   same grid over ALL original points (collision test)
    float4* apts;                     // [B][max_points]  x, y, z, point index bits
    // per-scan resident data
    const float4* xyzi;
    double *tail_x, *tail_y, *tail_z;
    float* tail_i;
    unsigned* label;
    double *r, *el;
    unsigned short* col;
    int* pix;
    unsigned char* alive;
    unsigned long long *zraw, *obj_raw;
    double* smooth;
    unsigned *dmask, *vmask;
    ScanState* st;
    int *gate_update, *gate_try, *gate_apply, *gate_full, *gate_patch;
    int* cf_rect;                     // [B][4] rows r0..r1, cols c0..c1 (inclusive) close/fill must recompute
    // work lists of the current round (per sub-batch; k_ctrl re-arms the counters, k_update fills them): the scans that
    // re-project in full, and the (scan, tile) tasks of close/fill — so those kernels run a small persistent grid
    // instead of one CTA per (chunk, scan) / (tile, scan) of which all but a few exit at once
    // ordered early-out of the placement search (OD): the reference takes the FIRST feasible yaw that keeps min_points,
    // so road level / collision / occlusion first look at the first `cand_window` on-map candidates (in yaw order) and
    // only the scans that found nothing there (need2) look at the rest, in the same round
    int cand_window;                  // 0 = evaluate every candidate at once
    int* need2;                       // [B]
    int* work_cnt;                    // [4]: scans in full_list, tasks in cf_tasks
    int* full_list;                   // [B]
    int* cf_tasks;                    // [B][cf_tiles]: scan * cf_tiles + tile
    int cf_tiles, cf_tiles_x;         // close/fill tiles per image, per image row of tiles
    int force_full;                   // debug / test: always take the full re-projection path
    int *col_off, *col_idx;           // [B][cols+1], [B][max_points]: original points bucketed by azimuth bin
    // round control of ONE sub-batch.  The round number lives on the device (round_ctl[0], advanced by the last k_ctrl
    // CTA) so that the launch sequence of a round has constant arguments and can be replayed as a CUDA graph.
    int* active_count;                // [64][2] per round slot: unfinished scans, finished k_ctrl CTAs
    unsigned long long* host_word;    // [64] mapped pinned host words; slot = round & 63 gets (seq << 32 | unfinished scans)
    unsigned* round_ctl;              // [2]: round number, sequence number of round 0 (seq of round r = base + r)
    unsigned long long* stats;        // [R3D_N_STATS] counters: 0 full projections, 1 tries, 2 masks applied, 3 in-place patches,
                                      // 4 / 5 selections in the shared tile / global scratch, 6 prefilter survivors, 7 on-map
                                      // rotations, 8 max steps of a scan (walker), 9 candidate windows, 10 exact occlusion
                                      // counts, 11 in-walker full re-projections
    int* far_arr;                     // [B] any smoothed scene pixel beyond 500 m (od/ins:486 quirk)
    // scene boxes
    Box* boxes;            // [B][max_boxes]
    BoxTest* box_tests;    // [B][max_boxes]
    // maps
    const unsigned char* od_maps;     // concatenated
    const long long* od_map_off;      // [B*2]
    const int* od_map_dims;           // [B*2*4]
    const unsigned char* ss_map;      // sequence map (values 0..3)
    int ss_sx, ss_sy;
    long long ss_move_x, ss_move_y;
    const double* poses;              // [B][16]
    unsigned* occ_win;                // [B][map_window*map_window/32]
    unsigned* occ_cnt;                // [B][map_window^2] scene points per marked cell of the window (walker: incremental marks)
    int* occ_far;                     // [B][64]: count + cells marked occupied outside the window (numpy-wrapped indices)
    // schedule
    const int* counts;                // [B][C]
    const int* perms;                 // [B][E][C][tries]
    unsigned* unplaceable;            // [B][ceil(n_objects/32)]
    // object DB
    const ObjBox* obj;
    ObjBox* try_obj;                  // [B] record of the cut object each scan is trying (written by k_onmap)
    const double *obj_x, *obj_y, *obj_z;
    const float* obj_i;
    const unsigned* obj_label;
    const int* class_list_off;
    const int* class_list;
    const double *cos_k, *sin_k;      // [K+1]
    const double* radii_sq;           // [50]
    const int* radii_ok;              // [50]
    const ClassCfg* classes;
    // candidates of the current try
    unsigned char* cand_flags;        // [B][K+1]  bit0 on map, bit1 road level found, bit2 collision
    double* cand_level;               // [B][K+1]
    int* cand_v;                      // [B][K+1]
    unsigned short* cand_list;        // [B][K+1] compacted rotations the next placement stage works on
    int* n_list;                      // [B]
    unsigned* tickets;                // [B][4]  "last CTA done" counters of the staged kernels (zeroed by k_ctrl)
    int* feas;                        // [B][K]
    int* occ_pix;                     // [B][OCC_G][max_obj_points] scratch
    int* sel_pix;                     // [B][max_obj_points]  scratch of k_select_emit for objects too large for shared memory
    unsigned long long* sel_keys;     // [B][sel_key_cap]
    double* sel_r;                    // [B][max_obj_points]
    int sel_key_cap;
    // outputs
    int* inserted;                    // [B][E][4]
    double* inserted_box;             // [B][E][8]
    float* check;                     // [B][max_inserted][5]
    int* chunk_cnt;                   // [B][max_chunks] live points per CHUNK of the working cloud (output compaction)
    int max_chunks;
    long long* out_count;             // [B] rows per scan ; out_off [B+1]
    long long* out_off;
    long long* check_off;
    float4* out_xyzi;
    unsigned* out_label;
    float* out_check;
    const float* world;               // [B][8] world augmentation (fx, fy, theta, c, s, k, 0, 0) of the output; NULL = off
};

// The world transform of r3d_world_aug (include/real3d_b200.h) on one point: flip, rotate, scale, in float32 without
// contraction, so that a host restatement reproduces it bit for bit
struct WorldXf { bool fx, fy; float c, s, k; };
__device__ __forceinline__ WorldXf world_xf(const float* w) {
    return WorldXf{w[0] != 0.f, w[1] != 0.f, w[3], w[4], w[5]};
}
__device__ __forceinline__ void world_point(const WorldXf& t, float& x, float& y, float& z) {
    const float x1 = t.fy ? -x : x, y1 = t.fx ? -y : y;
    x = __fmul_rn(__fsub_rn(__fmul_rn(t.c, x1), __fmul_rn(t.s, y1)), t.k);
    y = __fmul_rn(__fadd_rn(__fmul_rn(t.s, x1), __fmul_rn(t.c, y1)), t.k);
    z = __fmul_rn(z, t.k);
}

#define R3D_N_STATS 40
#ifndef R3D_OCC_G
#define R3D_OCC_G 8
#endif
constexpr int OCC_G = R3D_OCC_G;        // CTAs per scan in the occlusion-count kernel (8: +3.6 % over 16 with 8 engines in flight)
constexpr int OCC_FAR_CAP = 63;          // semseg: occupied map cells outside the per-scan bit window (see adjust_map_point)
constexpr double kFix = 1099511627776.0;   // 2^40 fixed point for the order-independent road-level sum

// thread `tid` (0 .. OCC_FAR_CAP) clears its entry of scan b's far-cell set
__device__ __forceinline__ void occ_far_clear(const EngineDev& e, int b, int tid) {
    if (tid <= OCC_FAR_CAP) e.occ_far[(size_t)b * (OCC_FAR_CAP + 1) + tid] = tid == 0 ? 0 : -1;
}

__device__ __forceinline__ void load_xyz(const EngineDev& e, int b, int p, int n0, double& x, double& y, double& z) {
    if (p < n0) {
        const float4 v = __ldg(&e.xyzi[(size_t)b * e.max_points + p]);
        x = (double)v.x; y = (double)v.y; z = (double)v.z;
    } else {
        const size_t t = (size_t)b * e.max_inserted + (p - n0);
        x = e.tail_x[t]; y = e.tail_y[t]; z = e.tail_z[t];
    }
}

}  // namespace r3d
