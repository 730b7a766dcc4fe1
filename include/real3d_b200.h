/* real3d_b200 — C ABI of the B200-native Real3D-Aug hot path (placement search + spherical occlusion + insertion).
 *
 * The reference (ctu-vras/pcl-augmentation) is pure Python with no FFI; its de-facto operator interface is the set
 * of module-level functions `insertion.py` star-imports (SURVEY.md §8b).  Each entry point below names the reference
 * function(s) it replaces.  Conventions: plain pointers and sizes only; every function returns 0 on success or a
 * negative error code (text via r3d_last_error()); outputs are caller-allocated; no ownership transfer; the
 * "primitive" calls are re-entrant per CUDA stream and take DEVICE pointers; the "engine" calls take HOST pointers
 * (they own the staging, the H2D/D2H copies and the device-resident state of a batch of scans).
 *
 * Row layouts are the reference's: a working point row is 9 float64
 *   [x, y, z, r, azimuth, elevation, intensity, label, pix_id]      (add_space_for_spherical, od/ins:55-65)
 * with od/ins = object_detection/Real3DAug/insertion.py, od/fs = .../tools/find_spot.py, cb = .../tools/cut_bbox.py,
 * cl = .../tools/closing.py, ss/... = the semantic_segmentation twins.
 */
#ifndef REAL3D_B200_H
#define REAL3D_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define R3D_OK 0
#define R3D_ERR_CUDA (-1)
#define R3D_ERR_ARG (-2)
#define R3D_ERR_ASSERT (-3)   /* the reference would have raised AssertionError (od/ins:111-113) */
#define R3D_ERR_INDEX (-4)    /* the reference would have raised IndexError (od/ins:410, < MAX_NUM_TRIES samples) */
#define R3D_ERR_CAPACITY (-5)

#define R3D_MAX_CLASSES 16
#define R3D_MAX_SURFACE 8
#define R3D_NUM_RADII 50
#define R3D_BOX_DOUBLES 16 /* cx cy cz(bottom) m00..m22(row-major) length width height reach */

typedef void* r3d_stream; /* cudaStream_t */

int r3d_version(void);
const char* r3d_last_error(void);
/* number of kernels this library has launched in this process (bench.py's gpu_launches) */
int64_t r3d_launch_count(void);

/* ------------------------------------------------------------------------------------------------ primitives */

/* fill_spherical (od/ins:68-82, ss/ins:67-81): r, azimuth, elevation of n working rows written in place to columns
 * 3..5; minmax_out[0] = max elevation, minmax_out[1] = min elevation (device, 2 doubles). */
int r3d_fill_spherical(double* rows9, int64_t n, double* minmax_out, r3d_stream stream);

/* geometrical_front_view (od/ins:85-130): spherical z-buffer.  train/label are num_row*num_col float64 (device);
 * pix_id = row * pix_stride + col goes to column 8 (pix_stride = the reference's module global NUMCOLUMN).
 * sample != 0 skips rows outside the elevation range (od/ins:108-109); otherwise an out-of-range bin sets
 * *status_out (device int) to R3D_ERR_ASSERT.  zbuf_scratch: num_row*num_col uint64 (device). */
int r3d_project_zbuffer(double* rows9, int64_t n, int num_row, int num_col, int pix_stride, double max_el,
                        double min_el, int sample, double* train_out, double* label_out, uint64_t* zbuf_scratch,
                        int* status_out, r3d_stream stream);

/* smooth_out + class_closing (cl:9-62): 5x3 closing of the occupancy and neighbour-mean hole fill.
 * closed_out (optional, may be NULL): the uint8 0/255 image class_closing returns. */
int r3d_close_fill(const double* train_in, const double* label_in, int num_row, int num_col, double* train_out,
                   double* label_out, uint8_t* closed_out, r3d_stream stream);

/* cut_bounding_box (cb:7-68): mask_out[i] = 1 iff point i (x,y,z = first three doubles of a row of row_stride
 * doubles) is strictly inside the box (R3D_BOX_DOUBLES doubles, host pointer). */
int r3d_cut_bounding_box(const double* rows, int64_t n, int row_stride, const double* box_host, uint8_t* mask_out,
                         r3d_stream stream);

/* rotate_bounding_box (od/fs:97-102, ss/fs:72) + the z move of correct_height (od/fs:167): in place on rows of
 * row_stride doubles (device): x' = c x - s y, y' = s x + c y, z' = z + dz. */
int r3d_transform_points(double* rows, int64_t n, int row_stride, double cos_t, double sin_t, double dz,
                         r3d_stream stream);

/* correct_height's growing-radius road-level search (od/fs:149-164, ss/fs:118-144) around (cx, cy) over rows whose
 * column label_col is one of labels[] and whose z > -3.  rows: device; labels, radii tables, outputs: host;
 * scratch3: 3 uint64 on the device.  Blocks until the result is on the host. */
int r3d_road_level(const double* rows, int64_t n, int row_stride, int label_col, const int32_t* labels, int n_labels,
                   double cx, double cy, const double* radii_sq, const int32_t* radii_ok, uint64_t* scratch3,
                   double* level_out, int32_t* ok_out, r3d_stream stream);

/* addjust_map_2 (ss/ins:202-224): map cells (value != 0) holding a working row with z < 1.5 and a label outside
 * ground_labels become 4.  rows9, map_dev (size_x * size_y float64): device; pose (4x4 row-major), labels: host. */
int r3d_adjust_map(const double* rows9, int64_t n, const double* pose16_host, int64_t move_x, int64_t move_y,
                   const int32_t* ground_labels, int n_ground, double* map_dev, int size_x, int size_y,
                   r3d_stream stream);

/* ------------------------------------------------------------------- stream-level placement / occlusion / insertion */
/* The stages of find_possible_places and of the occlusion / insertion step as re-entrant calls on DEVICE pointers
 * (caller-allocated outputs, no hidden state; the batched engine below is the fast path for many scans).
 *
 * r3d_place_candidates — A5 + A6 + A7 (od/fs:263-285, ss/fs:229-250) for the yaw_steps candidates of ONE cut object,
 * visited in order (the semseg map test of candidate k sees the z shift of the last candidate that passed and found a
 * road level, ss/fs:146-147).  obj_rows: m rows of row_stride doubles (x y z first); box8_host: cx cy cz(bottom) m00 m10
 * length width height; cos_k / sin_k: yaw_steps + 1 doubles (device), candidate k turns the object by k steps about
 * the sensor z axis.  task 0 (OD): map = uint8 {0, 1} size_x x size_y, move = (min_x, min_y), od/fs:267-279; task 1
 * (semseg): map = uint8 values 0..4 (after r3d_adjust_map), move = map move, pose16_host = lidar -> world,
 * map_ok_mask bit v = value v allowed (ss/fs:235-248).  ground_rows5: the ORIGINAL scan as n_ground x 5 float64
 * (x y z intensity label) for correct_height (od/fs:138-172); surface_labels (host): labels it accepts.
 * Outputs (device): flags_out[k] bit0 = on the map, bit1 = road level found; level_out[k] = road level. */
int r3d_place_candidates(const double* obj_rows, int64_t m, int32_t row_stride, const double* box8_host, int32_t yaw_steps,
                         const double* cos_k, const double* sin_k, int32_t task, const uint8_t* map, int32_t size_x,
                         int32_t size_y, int64_t move_x, int64_t move_y, const double* pose16_host, uint32_t map_ok_mask,
                         const double* ground_rows5, int64_t n_ground, const int32_t* surface_labels, int32_t n_surface,
                         const double* radii_sq_host, const int32_t* radii_ok_host, uint8_t* flags_out, double* level_out,
                         r3d_stream stream);

/* r3d_obb_collide — check_bounding_box (od/fs:109-135, ss/fs:79-104) for n_cand candidate placements at once:
 * collide_out[k] = 1 iff (i) an obstacle scene point lies strictly inside candidate k's box or (ii) one of candidate
 * k's object points lies strictly inside a scene box.  scene_rows9: n x 9 working rows (label = column 7);
 * scene_boxes / cand_boxes: R3D_BOX_DOUBLES each; obj_rows: the object's points BEFORE the candidate transform;
 * cand4[k] = {cos, sin, dz, 0}: candidate k's points are (c x - s y, s x + c y, z + dz).
 * mode 0 (OD): obstacle = label == 1 (od/fs:121), pedestrian != 0 keeps only points with z >= box bottom + 0.1
 * (od/fs:123); mode 1 (semseg): obstacle = label not in ok_labels (host, ss/fs:92-93). */
int r3d_obb_collide(const double* scene_rows9, int64_t n, const double* scene_boxes, int32_t n_boxes, const double* obj_rows,
                    int64_t m, int32_t row_stride, const double* cand4, const double* cand_boxes, int32_t n_cand, int32_t mode,
                    int32_t pedestrian, const int32_t* ok_labels, int32_t n_ok, uint8_t* collide_out, r3d_stream stream);

/* r3d_occlude_mask — od/ins:486-501: vis_px = obj_smooth < scene_smooth (strict; both num_pix float64 images as
 * r3d_close_fill returns them); scene_keep[i] = 0 iff the scene row's pix_id (column 8) is in vis_px; obj_keep[j] = 1
 * iff the object row's pix_id is >= 0 and in vis_px; counts_out (device int32[2]) = {scene rows removed, object rows
 * kept}; vis_px: num_pix uint8 (device, output). */
int r3d_occlude_mask(const double* scene_rows9, int64_t n, const double* obj_rows9, int64_t m, const double* scene_smooth,
                     const double* obj_smooth, int32_t num_pix, uint8_t* scene_keep, uint8_t* obj_keep, uint8_t* vis_px,
                     int32_t* counts_out, r3d_stream stream);

/* r3d_compact_insert — od/ins:545: out = the kept scene rows in order, then the kept object rows in (pix_id, index)
 * order (the order the reference's per-pixel loop appends them).  out_rows9: capacity n + m rows; n_out (device
 * int64[2]) = {rows written, of which scene rows}; sort_scratch: device uint64[scratch_len >= next_pow2(m)]. */
int r3d_compact_insert(const double* scene_rows9, const uint8_t* scene_keep, int64_t n, const double* obj_rows9,
                       const uint8_t* obj_keep, int64_t m, double* out_rows9, int64_t* n_out, uint64_t* sort_scratch,
                       int64_t scratch_len, r3d_stream stream);

/* ------------------------------------------------------------------------------------------------- rich maps */
/* object_detection/rich_map/single_drivable_area_map.py:123-194, batched over frames (all pointers: device).
 * xyzi: total x 4 float32, labels: total uint32 (semantic label & 0xFFFF), point_offsets: n_scans + 1.
 * Step 1 writes dims[scan] = {size_x, size_y, min_x, min_y} (1 m cells over the xy extent of ALL points, int()
 * truncation toward zero, :123-133).  The caller turns the sizes into cell offsets (map_offsets[scan], n_scans + 1) and
 * step 2 writes the road map (road points rasterised, closing(disk(4)), :136-161) and the pedestrian-area map
 * (8-neighbour ring of the road, dilation(disk(2)), :164-193) as uint8 {0, 1}, size_x * size_y cells each, row-major
 * [x][y]; scratch: 2 * total_cells bytes. */
int r3d_rich_map_od_extents(const float* xyzi, const int64_t* point_offsets, int32_t n_scans, int32_t* dims, r3d_stream stream);
int r3d_rich_map_od_build(const float* xyzi, const uint32_t* labels, const int64_t* point_offsets, int32_t n_scans,
                          uint32_t road_label, const int32_t* dims, const int64_t* map_offsets, int64_t total_cells,
                          uint8_t* road_out, uint8_t* ped_out, uint8_t* scratch, r3d_stream stream);

/* semantic_segmentation/rich_map/drivable_area_map.py:122-206: ONE map per sequence, built from frames that may be
 * fed in several calls (all pointers: device).  xyzi / labels / point_offsets as above; poses: n_frames x 16 float64
 * (row-major 4 x 4 lidar -> world, what SemanticKITTI.create_transform_matrix returns); max_points: the largest frame.
 * Step 1, r3d_rich_map_ss_extents: world-frame xy extent of all points (:130-146).  ext_state: 4 uint64 carried between
 * calls (first_call != 0 resets it); if out5 != NULL it receives {min_x, min_y, size_x, size_y, any_point} with
 * min = int(floor(min)), max = int(max) + 1 (:158-166).
 * Step 2, r3d_rich_map_ss_raster: the surface points of the frames in order (:172-200) into keymap (size_x * size_y
 * uint64, zeroed by the caller before the first call).  surface_labels[i] belongs to map class surface_classes[i]
 * (1 road: written unless the cell holds 3; 2 parking: likewise; 3 sidewalk: sticky); order_base = number of points
 * of the frames rasterised by earlier calls.  *error_flag becomes 1 where the reference's assert (:190) would fire,
 * 2 where it would raise IndexError.
 * Step 3, r3d_rich_map_ss_finalize: keymap -> map_out uint8 {0, 1, 2, 3}, row-major [x][y]. */
int r3d_rich_map_ss_extents(const float* xyzi, const int64_t* point_offsets, const double* poses, int32_t n_frames,
                            int32_t max_points, int32_t first_call, uint64_t* ext_state, int64_t* out5, r3d_stream stream);
int r3d_rich_map_ss_raster(const float* xyzi, const uint32_t* labels, const int64_t* point_offsets, const double* poses,
                           int32_t n_frames, int32_t max_points, const int32_t* surface_labels,
                           const int32_t* surface_classes, int32_t n_surface, int64_t min_x, int64_t min_y, int32_t size_x,
                           int32_t size_y, int64_t order_base, uint64_t* keymap, int32_t* error_flag, r3d_stream stream);
int r3d_rich_map_ss_finalize(const uint64_t* keymap, int64_t cells, uint8_t* map_out, r3d_stream stream);

/* ------------------------------------------------------------------------------------- cut-object database */
/* The point-in-box passes of object_detection/cut_object/object_cut_out.py:90-168 and
 * semantic_segmentation/cut_object/cut_out.py:103-157, batched over frames and boxes (all pointers: device).
 * xyzi / labels / point_offsets as above; boxes: n_boxes x R3D_BOX_DOUBLES, the boxes of frame f are
 * [box_offsets[f], box_offsets[f+1]) (at most 64 per frame: max_boxes_per_frame is the caller's promise).
 * Per box: keep_label >= 0 emits only the points carrying that label (cut_out.py:143), -1 any label, -2 none (the box is
 * only counted); use_drop != 0 additionally drops the labels of drop_labels (object_cut_out.py:150-152).
 * cameras: NULL or n_frames x 27 float64 = {M1 = V2C.T @ R0.T (4 x 3 row-major), P2 (3 x 4), image height, width, enabled}
 * for the field-of-view test of object_cut_out.py:144 (cutout.py:73-122).
 * r3d_cut_objects_count writes count_inside[box] (points strictly inside, cut_bbox.py:7-68), count_fov[box] (those the
 * camera sees), chunk_counts (scratch: n_boxes x ceil(max_points / 4096), kept for the write pass) and out_offsets
 * (n_boxes + 1: where the emitted points of each box start in the packed output).
 * r3d_cut_objects_write writes the emitted points of every box in their original order: out_xyzi (x, y, z, intensity
 * as read), out_labels, and optionally out_index (index of the point inside its frame). */
int r3d_cut_objects_count(const float* xyzi, const uint32_t* labels, const int64_t* point_offsets, int32_t n_frames,
                          int32_t max_points, const double* boxes, const int32_t* box_offsets, const int32_t* keep_label,
                          const int32_t* use_drop, int32_t n_boxes, int32_t max_boxes_per_frame, const double* cameras,
                          const int32_t* drop_labels, int32_t n_drop, int32_t* count_inside, int32_t* count_fov,
                          int32_t* chunk_counts, int64_t* out_offsets, r3d_stream stream);
int r3d_cut_objects_write(const float* xyzi, const uint32_t* labels, const int64_t* point_offsets, int32_t n_frames,
                          int32_t max_points, const double* boxes, const int32_t* box_offsets, const int32_t* keep_label,
                          const int32_t* use_drop, int32_t n_boxes, const int32_t* drop_labels, int32_t n_drop,
                          const int32_t* chunk_counts, const int64_t* out_offsets, float* out_xyzi, uint32_t* out_labels,
                          int32_t* out_index, r3d_stream stream);

/* --------------------------------------------------------------------------------------------------- engine */
/* Device-resident batched driver of the per-scan loop (od/ins:351-628, ss/ins:355-599): placement search
 * (find_possible_places od/fs:227-304, ss/fs:192-273), occlusion (od/ins:468-501), accept rule and insertion
 * (od/ins:530-561), sample scheduling (od/ins:386-428,587-614) and the output record (od/ds:76-109, ss/ds:72-106),
 * for many scans at once with the control flow on the device. */

typedef struct r3d_engine r3d_engine;

typedef struct r3d_class_cfg {
    int32_t min_points;   /* insertion.min_points[class] */
    int32_t map_sel;      /* OD: 0 = road map ("Road"), 1 = pedestrian-area map ("Sidewalk") (od/ins:434-441) */
    uint32_t map_ok_mask; /* semseg: bit v set iff map value v is in insertion.placement[class] (ss/fs:221,246) */
    int32_t pedestrian;   /* OD: class == 'Pedestrian' -> only scene points >= box bottom + 0.1 collide (od/fs:123) */
    int32_t n_surface;    /* labels the road-level search accepts: OD {labels.Road}; semseg placement_labels */
    int32_t surface[R3D_MAX_SURFACE];
} r3d_class_cfg;

typedef struct r3d_engine_cfg {
    int32_t task; /* 0 = object detection, 1 = semantic segmentation */
    int32_t rows, cols; /* range image (reference constants 112 x 1440, od/ins:21-22) */
    int32_t yaw_steps;  /* candidates per cut object (reference: 360, od/fs:263) */
    int32_t max_tries;  /* MAX_NUM_TRIES (od/ins:24) */
    int32_t n_classes;
    int32_t max_scans, max_points, max_inserted, max_boxes, max_events;
    int32_t road_label;                       /* OD: labels.Road (od/ins:354) */
    int32_t n_road_indexes;                   /* semseg addjust_map_2: ROAD_INDEXES (ss/ins:209) */
    int32_t road_indexes[R3D_MAX_SURFACE];
    int32_t map_window;                       /* semseg: side of the per-scan occupied-cell window (cells) */
    int32_t grid_half;                        /* road-level search grid: cells per half side (grid covers +-grid_half*grid_cell m) */
    double grid_cell;                         /* road-level search grid: cell size in metres (0 -> 0.5) */
    int32_t flags;                            /* bit0: re-project every slot in full (disable the in-place image patch);
                                                 bit1: launch the kernels of a round one by one instead of replaying the
                                                 round's CUDA graph;
                                                 bit2: evaluate every yaw candidate of a try at once (no ordered
                                                 early-out window; what r3d_engine_debug_candidates should see);
                                                 bit3: advance the batch with the STAGED round kernels (every stage of a
                                                 try is one batch-wide launch; needed by r3d_engine_debug_candidates)
                                                 instead of the default per-scan persistent walker (one CTA takes a scan
                                                 through all its slots and tries, ordered early exit per try);
                                                 bits 8-12 (staged rounds only): sub-batches advanced concurrently on
                                                 their own streams (1..16, 0 = default 4) */
    double radii_sq[R3D_NUM_RADII];           /* radius**2 of the growing search (od/fs:149-160), host-computed */
    int32_t radii_ok[R3D_NUM_RADII];          /* 0 where the pass's "radius > 5" check already fails */
    r3d_class_cfg classes[R3D_MAX_CLASSES];
} r3d_engine_cfg;

/* cut-object database (the role of glob(sample_path/<class>/ *.npz), sorted by name) */
typedef struct r3d_object_db {
    int32_t n_objects;
    const int64_t* point_offsets; /* n_objects + 1 */
    const double* points5;        /* total x 5 float64: x y z intensity label (object_cut_out.py:164-168) */
    const double* boxes;          /* n_objects x 8: cx cy cz(bottom) m00 m10 length width height (read_label_line) */
    const int32_t* class_index;   /* n_objects */
    const int32_t* class_list_offsets; /* n_classes + 1 */
    const int32_t* class_list;         /* object ids of each class in sorted-name order */
} r3d_object_db;

typedef struct r3d_batch {
    int32_t n_scans;
    const int64_t* point_offsets; /* n_scans + 1 */
    const float* xyzi;            /* total x 4 float32, as read from velodyne/ *.bin (od/ds:62) */
    const uint32_t* labels;       /* total, semantic label & 0xFFFF (od/ds:65); NULL when labels16 is given */
    const int32_t* box_offsets;   /* n_scans + 1 */
    const double* boxes;          /* total boxes x R3D_BOX_DOUBLES (scene annotations, extract_anno od/ins:133-157) */
    /* OD: two uint8 maps per scan (road, pedestrian area): dims[scan][map] = {size_x, size_y, min_x, min_y} */
    const int64_t* map_offsets;   /* (n_scans * 2) + 1, byte offsets into maps */
    const uint8_t* maps;
    const int32_t* map_dims;      /* n_scans x 2 x 4 */
    /* semseg: lidar->world 4x4 per scan (ss/ds:65-70); the sequence map is set with r3d_engine_set_ss_map */
    const double* poses;          /* n_scans x 16 */
    /* pre-drawn randomness (generate_seed od/ins:171-187, random.shuffle od/ins:400) */
    const int32_t* counts;        /* n_scans x n_classes */
    const int32_t* perms;         /* n_scans x n_events x n_classes x max_tries (object ids in class-list order) */
    int32_t n_events;
    const uint16_t* labels16;     /* total: the same labels packed to 16 bits (they are & 0xFFFF) — 2 instead of 4 bytes
                                     per point over PCIe; widened on the device */
    const uint8_t* labels1;       /* object detection only, (total + 7) / 8 bytes, used when labels and labels16 are NULL:
                                     bit i (little-endian bit order, i = index into the packed points of the batch) = point i
                                     carries the Road label.  The reference collapses the labels to {Road, 1} itself before
                                     the loop (od/ins:353-355), so one bit per point is all the OD path reads: 1/8 byte
                                     instead of 2 bytes per point over PCIe; expanded to {road_label, other} on the device */
} r3d_batch;

typedef struct r3d_batch_result {
    /* all host, caller-allocated; capacities given by the caller */
    int64_t* out_offsets;   /* n_scans + 1: rows of scan s are out_xyzi[out_offsets[s] .. out_offsets[s+1]) */
    float* out_xyzi;        /* capacity_points x 4: velodyne/<frame>.bin (od/ds:86-88) */
    uint32_t* out_labels;   /* capacity_points: labels/<frame>.label (ss/ds:82-84); may be NULL */
    int64_t capacity_points;
    int64_t* check_offsets; /* n_scans + 1 */
    float* check_xyzil;     /* capacity_check x 5: check/<frame>.bin rows x y z intensity label (ss/ds:76,86-88) */
    int64_t capacity_check;
    int32_t* n_inserted;    /* n_scans */
    int32_t* inserted;      /* n_scans x max_events x 4: object id, rotation (yaw step index), class index, visible points */
    double* inserted_box;   /* n_scans x max_events x 8: cx cy cz m00 m10 length width height of the placed box */
    int32_t* status;        /* n_scans: 0 or a negative R3D_ERR_* */
    int32_t* rounds;        /* 1: device rounds the batch took */
    uint16_t* out_labels16; /* capacity_points, alternative to out_labels: the same labels as 16-bit values (they are & 0xFFFF,
                               od/ds:65) — 2 instead of 4 bytes per point over PCIe; may be NULL */
} r3d_batch_result;

int r3d_engine_create(const r3d_engine_cfg* cfg, r3d_engine** out);
int r3d_engine_destroy(r3d_engine* eng);
int r3d_engine_set_yaw_tables(r3d_engine* eng, const double* cos_k, const double* sin_k); /* yaw_steps + 1 each */
int r3d_engine_set_objects(r3d_engine* eng, const r3d_object_db* db);
int r3d_engine_set_ss_map(r3d_engine* eng, const uint8_t* map, int32_t size_x, int32_t size_y, int64_t move_x,
                          int64_t move_y);
/* host -> device copy of a batch (async on the engine stream) + device-side preparation (A1/A2 spherical cache) */
int r3d_engine_load_batch(r3d_engine* eng, const r3d_batch* batch);
/* re-arm the already resident batch (alive flags, tails, scheduling state) without touching host memory */
int r3d_engine_reset_batch(r3d_engine* eng);
/* re-arm the resident batch; from_raw_points != 0 repeats the WHOLE device path from the resident float4 points
 * (spherical ingest A1/A2, spatial indices) — what a timed device-resident step must include */
int r3d_engine_rearm_batch(r3d_engine* eng, int from_raw_points);
/* run every scan of the batch to completion on the device and compact the outputs (device-resident) */
int r3d_engine_run(r3d_engine* eng);
/* device -> host copy of the results of the last run */
int r3d_engine_fetch(r3d_engine* eng, r3d_batch_result* result);
/* blocking wait for the engine stream */
/* Number of contiguous sub-batches r3d_engine_run advances concurrently, each on its own stream (1..8).  1 runs the
 * rounds strictly one kernel after the other (what the per-kernel CUDA-event profile needs). */
int r3d_engine_set_sub_batches(r3d_engine* eng, int n_sub);
/* r3d_engine_run in two (or more) calls: returns with *still_running = 1 as soon as at most `stop_at` scans of the batch
 * are unfinished (their rounds stay in flight); call again (stop_at = 0) to finish.  Lets a caller that serialises the
 * busy part of several engines' runs on one GPU overlap one engine's tail with the next engine's head. */
int r3d_engine_run_until(r3d_engine* eng, int stop_at, int* still_running);
int r3d_engine_sync(r3d_engine* eng);
/* total output rows of the last run (valid after r3d_engine_run + r3d_engine_sync) */
int r3d_engine_output_rows(r3d_engine* eng, int64_t* total_points, int64_t* total_check);
/* The packed outputs of the last run where they are, in device memory, for a consumer on the same GPU (a training
 * step that takes the augmented clouds without a round trip over PCIe): out_xyzi (total_points x 4 float32, the
 * velodyne rows of tools/datasets.py:86-93), out_labels (total_points uint32), check (total_check x 5 float32); the
 * per-scan row offsets go to the caller's HOST arrays (n_scans + 1 each, may be NULL).  Waits for the run; the
 * pointers stay valid until the engine is re-armed, loaded or run again. */
int r3d_engine_output_device(r3d_engine* eng, const float** out_xyzi, const uint32_t** out_labels, const float** check,
                             int64_t* out_offsets_host, int64_t* check_offsets_host);

/* per-kernel device time of the runs since the last reset, measured with CUDA events on the engine stream.
 * names_out: caller buffer receiving '\n'-separated kernel names; ms_out / launches_out: up to max_kernels entries. */
int r3d_engine_profile_enable(r3d_engine* eng, int on);
int r3d_engine_profile_read(r3d_engine* eng, char* names_out, int names_cap, double* ms_out, int64_t* launches_out,
                            int max_kernels, int* n_kernels_out);

/* find_possible_places (od/fs:227-304, ss/fs:192-273) for ONE cut object against an arbitrary current scene.
 * scene_rows9: host n_rows x 9 float64 working rows of the CURRENT scene (collision test, od/fs:120-127; semseg also
 * the occupied map cells of addjust_map_2); the scan's ORIGINAL points (road level), boxes, maps and pose come from
 * the loaded batch.  flags_out[k] (yaw_steps+1): bit0 on map, bit1 road level found, bit2 collision;
 * box_out[k] (yaw_steps+1 x 5): cx cy road-level m00 m10 of candidate k; xyz_out (optional): for the feasible
 * candidates in rotation order, n_points x 3 float64 each (capacity xyz_capacity candidates); *n_feasible_out.
 * Re-arms the batch state (run r3d_engine_reset_batch before the next r3d_engine_run). */
int r3d_engine_probe_places(r3d_engine* eng, int scan, int object_id, const double* scene_rows9, int64_t n_rows,
                            uint8_t* flags_out, double* box_out, double* xyz_out, int xyz_capacity,
                            int32_t* n_feasible_out);

/* gated scan-launch counters since the last r3d_engine_profile_enable: out8 = {scans re-projected in full, cut
 * objects tried, vis_px masks applied, scans patched in place, selections in the shared-memory tile, selections in
 * the global scratch image, 0, 0} — the "units one launch processes" of the roofline arithmetic */
int r3d_engine_stats(r3d_engine* eng, uint64_t* out8);
/* the first n (<= 32) counters: the 8 above, then {max steps of one scan in the last run, candidate windows evaluated,
 * exact occlusion counts (candidates the two-sided bound could not decide), full re-projections inside the walker,
 * 4 unused}, then the walker's phase clocks in SM cycles summed over all scans: {scheduling step, slot update, try
 * set-up + prefilter, placement windows, occlusion counts, selection + insertion, whole walk}, then finer clocks:
 * {on-map stage, road-level warps, collision warps, road-level searches, collision tests, mask apply, z-buffer patch,
 * close/fill} */
int r3d_engine_stats_ex(r3d_engine* eng, uint64_t* out, int n);
/* per scan of the last run (walker execution model): SM cycles its CTA lived and the cut objects it tried — the spread
 * between scans is what resident batches have to fill (DESIGN.md section 4.3) */
int r3d_engine_walk_profile(r3d_engine* eng, int64_t* cycles, int32_t* tries, int n);
/* the engine's cudaStream_t (so callers can bracket work with their own CUDA events) */
void* r3d_engine_stream(r3d_engine* eng);

/* ------------------------------------------------------------------------------- resident dataset (online) */
/* A dataset laid out in device memory, owned by the caller, from which r3d_engine_load_resident gathers batches
 * without any per-point host -> device traffic.  Device arrays (scan i of the store):
 *   xyzi [point_offsets[i] .. point_offsets[i+1]) x 4 float32 (16-byte aligned), labels the same rows as uint16
 *   (semantic label & 0xFFFF); boxes [box_offsets[i] .. box_offsets[i+1]) x R3D_BOX_DOUBLES (the records of
 *   r3d_batch.boxes); OD: maps / map_offsets (n_scans * 2 + 1, byte offsets into maps) / map_dims (n_scans x 2 x 4) in
 *   the r3d_batch layout; semseg: poses (n_scans x 16).  h_point_offsets / h_box_offsets: HOST copies of the
 *   offsets (capacity checks and the per-batch maxima without a device read). */
typedef struct r3d_resident_store {
    int32_t n_scans;
    const float* xyzi;
    const uint16_t* labels;
    const int64_t* point_offsets;
    const double* boxes;
    const int32_t* box_offsets;
    const uint8_t* maps;
    const int64_t* map_offsets;
    const int32_t* map_dims;
    const double* poses;
    const int64_t* h_point_offsets;
    const int32_t* h_box_offsets;
} r3d_resident_store;

/* How r3d_engine_load_resident draws the class counts of a scan (the insertion keys of the YAML, generate_seed
 * od/ins:171-187): random != 0 -> number_of_object independent uniform class draws; otherwise fixed_counts[n_classes]
 * (number_of_classes). */
int r3d_engine_set_schedule_policy(r3d_engine* eng, int32_t random, int32_t number_of_object, const int32_t* fixed_counts);
/* Load the store scans indices[0 .. n) (HOST array; duplicates allowed) as the engine's batch and draw their schedules
 * on the device: class counts and, per (event, class), a uniformly random ordered head of min(max_tries, list length)
 * distinct sample indices followed by -1 (random.shuffle od/ins:400), from Philox4x32-10 keyed by (seed, epoch, store
 * index, event, class) — never by the position in the batch, so a scan's draws do not depend on how scans are batched
 * or sharded.  The draws are integer arithmetic on Philox words (and float32 steps with one rounding each for the world
 * parameters), pinned bit for bit by the numpy restatement oracle/online_draws.py.  The device draw takes max_tries <=
 * 4266 (its shared memory, 48 bytes per try, within 200 KiB); a larger max_tries is R3D_ERR_CAPACITY here and works on
 * the host path.  Input errors are reported before anything is enqueued.  The only host -> device copy is the index list;
 * everything else is enqueued on the engine stream.  The OD maps are read from the store in place (keep it alive while
 * the batch is in use). */
int r3d_engine_load_resident(r3d_engine* eng, const r3d_resident_store* store, const int32_t* indices, int32_t n,
                             uint64_t seed, uint64_t epoch);
/* r3d_engine_set_ss_map on a map already in DEVICE memory (no copy; the engine only reads it; keep it alive). */
int r3d_engine_set_ss_map_device(r3d_engine* eng, const uint8_t* map, int32_t size_x, int32_t size_y, int64_t move_x,
                                 int64_t move_y);
/* device -> host copy of the schedule tables of the loaded batch: counts (n x n_classes), perms (n x *n_events x
 * n_classes x max_tries; may be NULL), *n_events. */
int r3d_engine_schedule_read(r3d_engine* eng, int32_t* counts, int32_t* perms, int32_t* n_events);
/* The inserted objects of the last run in DEVICE memory (the r3d_engine_output_device pattern, but enqueued on the
 * engine stream without a host wait): n_inserted (n), inserted (n x max_events x 4, as r3d_batch_result.inserted),
 * inserted_box (n x max_events x 8, likewise) and box7 (n x max_events x 7 float32: x, y, z_bottom, length, width,
 * height, yaw = atan2(m10, m00) in the lidar frame; rows past n_inserted are 0).  Valid until the next load / run. */
int r3d_engine_inserted_device(r3d_engine* eng, const int32_t** n_inserted, const int32_t** inserted,
                               const double** inserted_box, const float** box7);

/* World augmentation of resident batches: the random_world_flip / random_world_rotation / random_world_scaling steps
 * that detection recipes run after GT insertion, applied to the points and boxes of each scan together.  Per scan b
 * one Philox4x32-10 call (key = the schedule key of (seed, epoch), counter = (0, 0xFFFFFFFF, store index, epoch low
 * word), a stream the schedule draws never use) gives four 24-bit uniforms u0..u3:
 *   fx = u0 < flip_x_prob, fy = u1 < flip_y_prob, theta = rot_max * (2 u2 - 1), k = scale_lo + (scale_hi - scale_lo) u3,
 *   c = cosf(theta), s = sinf(theta).
 * A point (x, y, z) becomes, in float32 without contraction: x1 = fy ? -x : x, y1 = fx ? -y : y (flip along x negates
 * y, flip along y negates x), x' = (c x1 - s y1) k, y' = (s x1 + c y1) k, z' = z k.  Intensity and labels are kept.
 * A box centre follows the same arithmetic, its dimensions are multiplied by k, and its heading h becomes -h (flip x),
 * then -(h + pi) (flip y), then h + theta, wrapped to [-pi, pi).  A scan's parameters depend on (seed, epoch, store
 * index) only, like its schedule. */
typedef struct r3d_world_aug {
    float flip_x_prob, flip_y_prob;  /* in [0, 1] */
    float rot_max;                   /* in [0, pi] */
    float scale_lo, scale_hi;        /* 0 < scale_lo <= scale_hi */
} r3d_world_aug;

/* The world augmentation of the following r3d_engine_load_resident calls (NULL: off).  While it is on, each resident
 * load draws world[n][8] = (fx, fy, theta, c, s, k, 0, 0) on the device and the run writes transformed output points
 * and check rows; with it off a resident load enqueues what it enqueues without this call.  r3d_engine_load_batch
 * never applies it. */
int r3d_engine_set_world_aug(r3d_engine* eng, const r3d_world_aug* policy);
/* DEVICE pointer to the [n][8] world parameters of the loaded batch; fails unless that batch was loaded by
 * r3d_engine_load_resident with the world augmentation on.  Valid until the next load. */
int r3d_engine_world_device(r3d_engine* eng, const float** params);
/* Detection targets of inserted objects (object detection engines): dims3 (HOST, n_objects x 3) is the unpadded KITTI
 * (l, w, h) of each cut object; class_target (HOST, n_classes) maps an insertion class to its target class id
 * (1-based, 0 = not a target). */
int r3d_engine_set_object_targets(r3d_engine* eng, const float* dims3, const int32_t* class_target);
/* Every ground-truth box of each augmented scan of the last run, as detection targets in DEVICE buffers the caller
 * owns: out_box7 [n][max_targets][7] float32 (x, y, z_center, dx, dy, dz, heading) in the engine's lidar frame,
 * out_class [n][max_targets] int32 (0 = padding), out_count [n]; rows past a scan's count are zero.  The scene boxes
 * come first, in store order, then the inserted objects in insertion order.  scene_box7 / scene_class (DEVICE) hold
 * one target record and class id per box record of the store (indexed like its boxes through box_offsets); a class
 * of 0 skips the box.  An inserted object's box is (cx, cy, cz_bottom + h / 2, l, w, h, atan2(m10, m00) - pi / 2 wrapped
 * to [-pi, pi)) from its inserted_box record and dims3.  With the world augmentation on, the boxes are transformed
 * as the points are.  Enqueued on the engine stream after the run.  Errors, reported before anything is enqueued: no
 * run yet, a batch not loaded by r3d_engine_load_resident, a semseg engine, no r3d_engine_set_object_targets, or
 * max_targets below a scan's kept scene boxes + max_events - 1.  To check the last one the engine reads scene_class
 * back to the host the first time it sees the array, and assumes its contents do not change afterwards. */
int r3d_engine_targets_device(r3d_engine* eng, const r3d_resident_store* store, const float* scene_box7,
                              const int32_t* scene_class, int32_t max_targets, float* out_box7, int32_t* out_class,
                              int32_t* out_count);

/* debug / parity taps on the resident state of one scan (device -> host), used by the tests */
int r3d_engine_debug_image(r3d_engine* eng, int scan, double* smooth_out /* rows*cols */);
int r3d_engine_debug_candidates(r3d_engine* eng, int scan, uint8_t* flags_out /* yaw_steps+1 */,
                                double* level_out /* yaw_steps+1 */, int32_t* visible_out /* yaw_steps+1 */);

#ifdef __cplusplus
}
#endif
#endif /* REAL3D_B200_H */
