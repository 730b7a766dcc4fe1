// Launchers of the resident-dataset kernels (r3d_resident.cu), called by r3d_engine_load_resident and
// r3d_engine_inserted_device in r3d_engine.cu.  All pointers are device pointers; everything is enqueued on `st`.
#pragma once
#include "r3d_engine.cuh"

namespace r3d {

struct SchedulePolicy {
    int random, number_of_object;
    int fixed[R3D_MAX_CLASSES];
};

// store rows of the scans idx[0 .. n) -> per-scan rows xyzi [n][max_points] and label [n][P]; OD labels collapse to
// {road_label, other} as k_expand_label_bits does, semseg labels widen as k_widen_labels does
void launch_gather_points(const r3d_resident_store& s, const int* idx, int n, int max_n0, float4* xyzi, int max_points,
                          unsigned* label, int P, int od, unsigned road_label, cudaStream_t st);
// per-scan metadata (n0, scene-box count, OD map offsets / dims or semseg pose) and the scene boxes (zero-padded to
// max_boxes) into boxes and boxes0
void launch_gather_meta(const r3d_resident_store& s, const int* idx, int n, int od, int* n0, int* nbox0, long long* map_off,
                        int* map_dims, double* poses, Box* boxes, Box* boxes0, int max_boxes, cudaStream_t st);
// Dynamic shared memory of k_draw_schedule for max_tries T (three int arrays of T per warp), and the largest T the
// device draw takes: 48 * T within 200 KiB, T <= 4266.  The bound also keeps the step j below 2^16, which the
// (j | attempt << 16) counter word of a head draw needs.
size_t draw_schedule_smem(int T);
constexpr int DRAW_MAX_TRIES = 4266;
// raises k_draw_schedule's dynamic shared memory limit on the current device to draw_schedule_smem(T) (never lowers
// it, so engines with different max_tries can share the device); T <= DRAW_MAX_TRIES
cudaError_t allow_draw_schedule_smem(int T);
// counts [n][C] and perms [n][E][C][T] of the scans idx[0 .. n) for (seed, epoch)
void launch_draw_schedule(const int* idx, int n, int E, int C, int T, const int* class_list_off, const SchedulePolicy& pol,
                          unsigned long long seed, unsigned long long epoch, int* counts, int* perms, cudaStream_t st);
// n_inserted [n] and the float32 boxes [n][E][7] of the last run
void launch_inserted_targets(const ScanState* sts, const double* inserted_box, int n, int E, int* n_inserted, float* box7,
                             cudaStream_t st);
// world [n][8] = (fx, fy, theta, c, s, k, 0, 0) of the scans idx[0 .. n) for (seed, epoch) (r3d_world_aug)
void launch_draw_world(const int* idx, int n, const r3d_world_aug& pol, unsigned long long seed, unsigned long long epoch,
                       float* world, cudaStream_t st);
// detection targets of the last run (r3d_engine_targets_device); world may be NULL
void launch_gt_targets(const int* idx, const int* box_off, const float* scene_box7, const int* scene_class, const ScanState* sts,
                       const int* inserted, const double* inserted_box, int E, const float* dims3, const int* class_target,
                       const float* world, int n, int max_targets, float* out_box7, int* out_class, int* out_count,
                       cudaStream_t st);
// Points of the output rows xyzi (scan b: rows out_off[b] .. out_off[b + 1], at most max_rows) inside the first
// min(count[b], cap) targets of box7 / cls / count (r3d_engine_target_points_device): points [n][max_targets] and
// point_gt per row; with min_points > 0 the targets below it are dropped in place and point_gt refers to the kept ones.
// remap: [n][cap + 1] scratch.  Dynamic shared memory: target_points_smem(cap), cap <= TARGET_POINTS_MAX_BOXES.
constexpr int TARGET_POINTS_MAX_BOXES = 2048;
size_t target_points_smem(int cap);
cudaError_t launch_target_points(const float4* xyzi, const long long* out_off, int n, int max_rows, float* box7, int* cls,
                                 int* count, int max_targets, int cap, int min_points, int* points, int* point_gt, int* remap,
                                 cudaStream_t st);

}  // namespace r3d
