// Host side of the batched Real3D-Aug engine: device memory, H2D/D2H staging, the per-round launch sequence and
// the C ABI declared in include/real3d_b200.h.
#include "r3d_engine_kernels.cuh"
#include "r3d_host.h"
#include "r3d_resident.h"

#include <cmath>
#include <chrono>
#include <cstdlib>
#include <thread>
#include <cstring>
#include <map>
#include <memory>
#include <string>
#include <vector>

using namespace r3d;

#define R3D_MAX_SUB 16
// the three full re-projection kernels and close/fill walk the work lists k_update wrote (all scans in round 0, a
// handful later): grids sized for "some scans", not for every (chunk, scan) / (tile, scan) pair
#define R3D_FULL_Y 32

namespace {

enum KernelId {
    KID_INGEST, KID_CTRL, KID_UPDATE, KID_CLEAR, KID_PROJECT, KID_CLOSEFILL, KID_ADJUST, KID_ONMAP, KID_HEIGHT, KID_COLLIDE,
    KID_GRID, KID_OCCL, KID_SELECT, KID_OUT, KID_MINMAX, KID_PROJECT0, KID_CLOSEFILL0, KID_CLEAR0, KID_MINMAX0, KID_WALK, KID_PREP, KID_SCATTER,
    KID_COUNT
};
const char* kKernelNames[KID_COUNT] = {
    "ingest_spherical", "ctrl", "update_mask_patch", "clear_images", "project_zbuffer", "close_fill", "adjust_map",
    "onmap", "road_level", "collide", "index_build", "occlusion_count", "select_emit", "compact_output", "minmax_elevation",
    // round 0 of a run re-projects every scan in full; later rounds only the scans whose elevation range moved
    "project_zbuffer_full", "close_fill_full", "clear_images_full", "minmax_elevation_full",
    // the per-scan persistent walker (one CTA per scan runs all the slots / tries of its scan) and its set-up
    "scan_walk", "walk_prepare",
    // fused streaming passes: ingest_spherical = A1 + A2 + index counts + z-buffer clear, index_build = scans + distance
    // transform, scatter_project = CSR scatter of the three indices + A3 (pix ids, z-buffer)
    "scatter_project"};

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    int alloc(size_t count) {
        release();
        n = count;
        if (count == 0) return R3D_OK;
        cudaError_t err = cudaMalloc((void**)&p, count * sizeof(T));
        if (err != cudaSuccess) { p = nullptr; return r3d_fail_cuda(err, "cudaMalloc"); }
        return R3D_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; n = 0; }
    ~DevBuf() { release(); }
};

}  // namespace

struct r3d_engine {
    r3d_engine_cfg cfg;
    EngineDev dev;
    cudaStream_t stream = nullptr;
    int n_scans = 0;
    int max_n0 = 0;
    int n_sms = 148;
    int device = 0;                              // every API call binds the calling thread to the engine's device first
    int n_sub = 4;                               // sub-batches advanced concurrently, each on its own stream
    cudaStream_t sub_stream[R3D_MAX_SUB] = {nullptr};
    cudaEvent_t sub_done[R3D_MAX_SUB] = {nullptr};
    cudaEvent_t ev_armed = nullptr;
    cudaEvent_t ev_wait = nullptr;               // blocking-sync event for host waits on the engine stream
    // state of a run in progress (r3d_engine_run_until may return before the batch is finished)
    struct Sub { int b0, n, round; bool done; long long left; unsigned seq_base; EngineDev d; cudaStream_t st; };
    Sub sub[R3D_MAX_SUB];
    // one round of a sub-batch (k_ctrl ... k_select_emit) captured as a CUDA graph: every argument is constant between
    // rounds (the round number lives on the device), so a round costs the host ONE launch instead of twelve
    struct RoundGraph { cudaGraphExec_t exec = nullptr; EngineDev d; int ns = 0, chunks_all = 0, task_ctas = 0, sel_pts = 0, kernels = 0; };
    RoundGraph round_graph[R3D_MAX_SUB];
    bool use_graphs = true, capturing = false;
    bool fresh = false;                          // ingest just ran: z-buffer / pix ids / elevation range of the originals are valid
    bool walked = false;                         // the last run used the walker (its step count is in h_offsets)
    bool staged = false;                         // true: the staged round kernels (debug / probe path); false: the per-scan walker
    bool run_active = false;
    int run_nsub = 0, run_done = 0, run_rounds = 0;
    bool objects_set = false, yaw_set = false, batch_loaded = false, ran = false;
    int last_rounds = 0;
    // the per-scan arrays of `dev` ([B][extent], allocated by per_scan()): device memory owned by the engine, and the
    // field's byte offset in EngineDev and per-scan byte stride, by which sub_view() moves it to a sub-batch
    struct PerScan { size_t field, stride; void* p; };
    std::vector<PerScan> scan_arrays;
    // batch-wide device buffers, and buffers the kernels do not see through EngineDev
    DevBuf<float4> out_xyzi;
    DevBuf<double> obj_x, obj_y, obj_z, cos_k, sin_k, radii_sq;
    DevBuf<float> obj_i, out_check;
    DevBuf<unsigned> obj_label, out_label, round_ctl;
    DevBuf<unsigned short> label16, out_label16;
    DevBuf<unsigned char> label1, od_maps, ss_map;
    DevBuf<int> active_count, perms, class_list_off, class_list, radii_ok, n0_arr, nbox0_arr;
    DevBuf<unsigned long long> stats;
    DevBuf<long long> pt_off, od_map_off, out_off, check_off;
    DevBuf<Box> boxes0;                          // the scene boxes as loaded (re-arm drops the inserted ones, device to device)
    DevBuf<ObjBox> obj;
    DevBuf<ClassCfg> classes;
    CUtensorMap zraw_tmap;            // [B][H][W] u64 z-buffer as a 3-D tiled tensor, box = one staged close/fill tile
    bool zraw_tmap_ok = false;
    std::vector<int> h_nbox0;                    // scene boxes per scan of the loaded batch
    unsigned long long* h_words = nullptr;   // mapped pinned: one word per round slot, written by k_ctrl
    unsigned long long* d_words = nullptr;   // device alias of h_words
    unsigned seq = 0;
    long long* h_offsets = nullptr;     // pinned, 2 * (max_scans + 1)
    // resident-dataset loads (r3d_engine_load_resident): schedule policy, the pinned index list and the event after its
    // copy (the list is rewritten only once the previous copy has left it), detection targets of the last run
    SchedulePolicy policy;
    bool policy_set = false;
    int* h_idx = nullptr;
    cudaEvent_t ev_idx = nullptr;
    DevBuf<int> idx_dev, n_ins_dev;
    DevBuf<float> box7;
    bool from_store = false;                     // the batch came from r3d_engine_load_resident (store indices in batch_idx)
    std::vector<int> batch_idx;
    // world augmentation (r3d_engine_set_world_aug): the policy, and whether the loaded batch drew its world[n][8]
    r3d_world_aug world_pol;
    bool world_on = false, world_loaded = false;
    DevBuf<float> world;
    // detection targets (r3d_engine_set_object_targets / r3d_engine_targets_device); kept scene boxes per store scan,
    // read back once per scene_class array
    DevBuf<float> obj_dims3;
    DevBuf<int> class_target;
    const int* kept_src = nullptr;
    std::vector<int> kept;
    // most targets a scan of the loaded batch can have (kept scene boxes + max_events), set by the batch's
    // r3d_engine_targets_device (0: not yet), and the [B][cap + 1] remap scratch of r3d_engine_target_points_device
    int targets_bound = 0;
    DevBuf<int> tp_remap;
    // profiling
    bool profile = false;
    double prof_ms[KID_COUNT] = {0};
    int64_t prof_launches[KID_COUNT] = {0};
    std::vector<std::pair<int, std::pair<cudaEvent_t, cudaEvent_t>>> pending_events;
    std::vector<cudaEvent_t> event_pool;

    // releases everything, also of an engine whose creation failed part way (null handles are skipped); the DevBuf
    // members are freed after this body, once the sub-batch streams are idle
    ~r3d_engine() {
        for (int i = 0; i < R3D_MAX_SUB; ++i) {
            if (sub_stream[i]) { cudaStreamSynchronize(sub_stream[i]); cudaStreamDestroy(sub_stream[i]); }
            if (sub_done[i]) cudaEventDestroy(sub_done[i]);
            if (round_graph[i].exec) cudaGraphExecDestroy(round_graph[i].exec);
        }
        for (const PerScan& a : scan_arrays) cudaFree(a.p);
        for (cudaEvent_t ev : event_pool) cudaEventDestroy(ev);
        for (cudaEvent_t ev : {ev_armed, ev_wait, ev_idx})
            if (ev) cudaEventDestroy(ev);
        if (h_words) cudaFreeHost(h_words);
        if (h_offsets) cudaFreeHost(h_offsets);
        if (h_idx) cudaFreeHost(h_idx);
        if (stream) cudaStreamDestroy(stream);
    }
};

namespace {

__global__ void k_box_tests(const Box* boxes, BoxTest* tests, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) tests[i] = make_box_test(boxes[i]);
}
// packed 16-bit labels (contiguous, per-scan offsets) -> the engine's u32 label rows
__global__ void k_widen_labels(const unsigned short* src, const long long* pt_off, unsigned* label, int P, int n_scans) {
    const int b = blockIdx.y;
    if (b >= n_scans) return;
    const long long o = pt_off[b] - pt_off[0];
    const int cnt = (int)(pt_off[b + 1] - pt_off[b]);
    const int p0 = blockIdx.x * CHUNK;
    for (int p = p0 + threadIdx.x; p < min(p0 + CHUNK, cnt); p += blockDim.x) label[(size_t)b * P + p] = src[o + p];
}
// one "is Road" bit per point (object detection) -> {road_label, some other label}
__global__ void k_expand_label_bits(const unsigned char* bits, const long long* pt_off, unsigned* label, int P, int n_scans,
                                    unsigned road_label) {
    const int b = blockIdx.y;
    if (b >= n_scans) return;
    const long long o = pt_off[b] - pt_off[0];
    const int cnt = (int)(pt_off[b + 1] - pt_off[b]);
    const int p0 = blockIdx.x * CHUNK;
    const unsigned other = road_label == 1u ? 2u : 1u;       // od/ins:353-355 relabels every non-Road point to 1
    for (int p = p0 + threadIdx.x; p < min(p0 + CHUNK, cnt); p += blockDim.x) {
        const long long i = o + p;
        label[(size_t)b * P + p] = ((bits[i >> 3] >> (i & 7)) & 1u) ? road_label : other;
    }
}
__global__ void k_narrow_labels(const unsigned* src, unsigned short* dst, long long n) {
    for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dst[i] = (unsigned short)src[i];
}
__global__ void k_set_round(unsigned* round_ctl, unsigned seq_base) { round_ctl[0] = 0u; round_ctl[1] = seq_base; }
__global__ void k_fill_u64(unsigned long long* p, size_t n, unsigned long long v) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = v;
}

struct Launcher {          // wraps every launch: launch counter + optional CUDA-event timing on the launching stream
    r3d_engine* eng;
    int kid;
    cudaStream_t st;
    cudaEvent_t a = nullptr, b = nullptr;
    Launcher(r3d_engine* e, int k, cudaStream_t stream = nullptr) : eng(e), kid(k), st(stream ? stream : e->stream) {
        if (eng->profile) {
            a = get_event(); b = get_event();
            cudaEventRecord(a, st);
        }
    }
    cudaEvent_t get_event() {
        if (!eng->event_pool.empty()) { cudaEvent_t ev = eng->event_pool.back(); eng->event_pool.pop_back(); return ev; }
        cudaEvent_t ev; cudaEventCreate(&ev); return ev;
    }
    ~Launcher() {
        if (eng->capturing) return;          // counted per graph launch
        r3d_count_launch();
        eng->prof_launches[kid] += 1;
        if (eng->profile) {
            cudaEventRecord(b, st);
            eng->pending_events.push_back({kid, {a, b}});
        }
    }
};

void drain_events(r3d_engine* eng) {
    for (auto& pe : eng->pending_events) {
        float ms = 0.f;
        cudaEventSynchronize(pe.second.second);
        cudaEventElapsedTime(&ms, pe.second.first, pe.second.second);
        eng->prof_ms[pe.first] += ms;
        eng->event_pool.push_back(pe.second.first);
        eng->event_pool.push_back(pe.second.second);
    }
    eng->pending_events.clear();
}

size_t occl_smem_bytes(const EngineDev& d) { return (size_t)d.dwords * sizeof(unsigned) + (size_t)(d.K + 2) * sizeof(unsigned short); }
constexpr int SEL_SMEM_PTS = 4096;       // object points k_select_emit keeps in shared memory; larger objects use global scratch
int next_pow2(int v) { int p = 1; while (p < v) p <<= 1; return p; }
// dynamic shared memory of k_select_emit: sort keys, ranges, object tile, pixel ids, dilation + visibility bits
size_t select_smem_bytes(int max_pts) {
    return (size_t)next_pow2(max_pts) * 8 + (size_t)max_pts * 8 + (size_t)SEL_TILE_PX * 8 + (size_t)max_pts * 4 +
           2 * (size_t)(SEL_TILE_PX / 32) * 4 + 16;
}

// Allocates the per-scan array `field` of eng->dev: B x `extent` elements, owned by the engine.  This is the only place
// that states a per-scan array's extent: sub_view() offsets every array allocated here by the same stride.  A field
// allocated again (a new object DB) frees its previous array.
template <class T>
int per_scan(r3d_engine* eng, T*& field, size_t extent) {
    const size_t at = (size_t)(reinterpret_cast<char*>(&field) - reinterpret_cast<char*>(&eng->dev));
    for (size_t i = 0; i < eng->scan_arrays.size(); ++i)
        if (eng->scan_arrays[i].field == at) {
            cudaFree(eng->scan_arrays[i].p);
            eng->scan_arrays.erase(eng->scan_arrays.begin() + i);
            break;
        }
    field = nullptr;
    void* p = nullptr;
    const cudaError_t err = cudaMalloc(&p, (size_t)eng->dev.B * extent * sizeof(T));
    if (err != cudaSuccess) return r3d_fail_cuda(err, "cudaMalloc");
    eng->scan_arrays.push_back({at, extent * sizeof(T), p});
    field = static_cast<T*>(p);
    return R3D_OK;
}

// the host fills some arrays the kernels only read (EngineDev declares them const)
template <class T> T* mut(const T* p) { return const_cast<T*>(p); }

// every API call first binds the calling thread to the engine's device; false for a null engine
bool bind(r3d_engine* eng) {
    if (!eng) return false;
    cudaSetDevice(eng->device);
    return true;
}

}  // namespace

#define TRY(x) do { int _rc = (x); if (_rc != R3D_OK) return _rc; } while (0)

// Wait for the engine stream WITHOUT spinning: the waits below cover millisecond-long transfers and whole runs, and a
// rank keeps several engine threads; cudaStreamSynchronize would burn a host core per waiting thread (8 ranks x 4
// pipelined engines on a 32-vCPU box starve the threads that launch the rounds).  A blocking-sync event sleeps instead.
static cudaError_t engine_wait(r3d_engine* eng) {
    if (!eng->ev_wait) {
        cudaError_t e = cudaEventCreateWithFlags(&eng->ev_wait, cudaEventBlockingSync | cudaEventDisableTiming);
        if (e != cudaSuccess) return e;
    }
    cudaError_t e = cudaEventRecord(eng->ev_wait, eng->stream);
    if (e != cudaSuccess) return e;
    return cudaEventSynchronize(eng->ev_wait);
}

// TMA descriptor of the z-buffer for k_close_fill_tma (r3d_closefill.cuh).  cuTensorMapEncodeTiled is a driver API entry:
// fetched through the runtime so that the library does not link against libcuda.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static bool make_zraw_tensor_map(CUtensorMap* tm, void* base, int W, int H, int B) {
    if (getenv("R3D_NO_TMA") || (W & 1) || ((uintptr_t)base & 15)) return false;       // row pitch must be a multiple of 16 bytes
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
        cudaGetLastError();
        return false;
    }
    const cuuint64_t dims[3] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B};
    const cuuint64_t strides[2] = {(cuuint64_t)W * 8, (cuuint64_t)W * H * 8};
    const cuuint32_t box[3] = {(cuuint32_t)CF_SW, (cuuint32_t)CF_SH, 1u};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return ((EncodeTiledFn)fn)(tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                               CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

extern "C" int r3d_engine_create(const r3d_engine_cfg* cfg, r3d_engine** out) {
    if (!cfg || !out) return r3d_fail(R3D_ERR_ARG, "r3d_engine_create: null argument");
    if (cfg->rows <= 0 || cfg->cols <= 0 || cfg->cols > 65535 || cfg->yaw_steps <= 0 || cfg->n_classes <= 0 ||
        cfg->n_classes > R3D_MAX_CLASSES || cfg->max_scans <= 0 || cfg->max_points <= 0 || cfg->max_inserted <= 0 ||
        cfg->max_tries <= 0 || cfg->max_events <= 0 || cfg->max_boxes <= 0 || (cfg->task != 0 && cfg->task != 1))
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_create: bad configuration");
    if (cfg->task == 1 && (cfg->map_window <= 0 || cfg->map_window % 32 != 0))
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_create: map_window must be a positive multiple of 32");
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
        return r3d_fail(R3D_ERR_CUDA, "r3d_engine_create: no CUDA device (this library has no CPU fallback)");
    std::unique_ptr<r3d_engine> owner(new r3d_engine());           // frees whatever was created if a step below fails
    r3d_engine* eng = owner.get();
    eng->cfg = *cfg;
    EngineDev& d = eng->dev;
    memset(&d, 0, sizeof(d));
    d.task = cfg->task; d.rows = cfg->rows; d.cols = cfg->cols; d.hw = cfg->rows * cfg->cols; d.K = cfg->yaw_steps;
    d.max_tries = cfg->max_tries; d.n_classes = cfg->n_classes; d.B = cfg->max_scans; d.max_points = cfg->max_points;
    d.max_inserted = cfg->max_inserted + (16 - (cfg->max_points + cfg->max_inserted) % 16) % 16;   // rows of P: 16-aligned
    d.P = cfg->max_points + d.max_inserted; d.max_boxes = cfg->max_boxes;
    d.max_events = cfg->max_events; d.road_label = cfg->road_label; d.n_road_indexes = cfg->n_road_indexes;
    d.map_window = cfg->task == 1 ? cfg->map_window : 32; d.dwords = (d.hw + 31) / 32;
    for (int i = 0; i < R3D_MAX_SURFACE; ++i) d.road_indexes[i] = cfg->road_indexes[i];
    d.step_rad = 2.0 * 3.14159265358979323846 / (double)cfg->yaw_steps;
    d.grid_cell = cfg->grid_cell > 0 ? cfg->grid_cell : 0.5;
    d.grid_inv_cell = (float)(1.0 / d.grid_cell);
    d.G = 2 * (cfg->grid_half > 0 ? cfg->grid_half : 200);
    d.force_full = (cfg->flags & 1) ? 1 : 0;
    d.cf_tiles_x = (d.cols + CF_TW - 1) / CF_TW;
    d.cf_tiles = d.cf_tiles_x * ((d.rows + CF_TH - 1) / CF_TH);
    d.cand_window = (cfg->flags & 4) ? 0 : 48;
    if (d.task != 0) d.cand_window = 0;          // semseg walks the yaws with a carried z shift (ss/fs:146-147): no window
    d.max_chunks = (d.P + CHUNK - 1) / CHUNK;
    if (d.max_points + d.max_inserted > (1 << APT_IDX_BITS)) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_create: more than 2^27 points per scan");
    std::vector<ClassCfg> cls(R3D_MAX_CLASSES);
    for (int c = 0; c < R3D_MAX_CLASSES; ++c) {
        const r3d_class_cfg& s = cfg->classes[c];
        cls[c].min_points = s.min_points; cls[c].map_sel = s.map_sel; cls[c].map_ok_mask = s.map_ok_mask;
        cls[c].pedestrian = s.pedestrian; cls[c].n_surface = std::min(std::max(s.n_surface, 0), R3D_MAX_SURFACE);
        for (int i = 0; i < R3D_MAX_SURFACE; ++i) cls[c].surface[i] = s.surface[i];
        cls[c].ok_slots = 0u;
    }
    d.n_surf_all = 0;
    for (int c = 0; c < cfg->n_classes; ++c)
        for (int i = 0; i < cls[c].n_surface; ++i) {
            int slot = -1;
            for (int j = 0; j < d.n_surf_all; ++j) if (d.surf_all[j] == cls[c].surface[i]) slot = j;
            if (slot < 0) {
                if (d.n_surf_all >= 15) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_create: more than 15 distinct surface labels");
                slot = d.n_surf_all; d.surf_all[d.n_surf_all++] = cls[c].surface[i];
            }
            cls[c].ok_slots |= 1u << slot;
        }
    eng->n_sub = (cfg->flags >> 8) & 31;
    if (eng->n_sub <= 0) eng->n_sub = 4;
    eng->n_sub = std::min(eng->n_sub, R3D_MAX_SUB);
    eng->use_graphs = !(cfg->flags & 2);
    eng->staged = (cfg->flags & 8) != 0;
    R3D_CUDA(cudaGetDevice(&eng->device));
    R3D_CUDA(cudaDeviceGetAttribute(&eng->n_sms, cudaDevAttrMultiProcessorCount, eng->device));
    // the round kernels (short, latency bound) run on high-priority streams; uploads, the one-off spherical ingest /
    // index builds and the output compaction of OTHER engines on the same GPU (ScanPipeline) must not sit in front of them
    int prio_least = 0, prio_greatest = 0;
    R3D_CUDA(cudaDeviceGetStreamPriorityRange(&prio_least, &prio_greatest));
    R3D_CUDA(cudaStreamCreateWithPriority(&eng->stream, cudaStreamNonBlocking, prio_least));
    for (int i = 0; i < R3D_MAX_SUB; ++i) {
        R3D_CUDA(cudaStreamCreateWithPriority(&eng->sub_stream[i], cudaStreamNonBlocking, prio_greatest));
        R3D_CUDA(cudaEventCreateWithFlags(&eng->sub_done[i], cudaEventDisableTiming));
    }
    R3D_CUDA(cudaEventCreateWithFlags(&eng->ev_armed, cudaEventDisableTiming));
    const size_t B = d.B, P = d.P, K1 = d.K + 1, GG = (size_t)d.G * d.G, MW2 = (size_t)d.map_window * d.map_window;
    TRY(per_scan(eng, d.xyzi, d.max_points)); TRY(per_scan(eng, d.tail_x, d.max_inserted)); TRY(per_scan(eng, d.tail_y, d.max_inserted));
    TRY(per_scan(eng, d.tail_z, d.max_inserted)); TRY(per_scan(eng, d.tail_i, d.max_inserted)); TRY(per_scan(eng, d.label, P));
    TRY(per_scan(eng, d.r, P)); TRY(per_scan(eng, d.el, P)); TRY(per_scan(eng, d.col, P)); TRY(per_scan(eng, d.pix, P));
    TRY(per_scan(eng, d.alive, P)); TRY(per_scan(eng, d.zraw, d.hw)); TRY(per_scan(eng, d.obj_raw, d.hw)); TRY(per_scan(eng, d.smooth, d.hw));
    eng->zraw_tmap_ok = make_zraw_tensor_map(&eng->zraw_tmap, d.zraw, d.cols, d.rows, (int)B);
    TRY(per_scan(eng, d.dmask, d.dwords)); TRY(per_scan(eng, d.vmask, d.dwords)); TRY(per_scan(eng, d.st, 1));
    TRY(per_scan(eng, d.gate_update, 1)); TRY(per_scan(eng, d.gate_try, 1)); TRY(per_scan(eng, d.gate_apply, 1));
    TRY(per_scan(eng, d.gate_full, 1)); TRY(per_scan(eng, d.gate_patch, 1)); TRY(per_scan(eng, d.cf_rect, 4));
    TRY(per_scan(eng, d.work_cnt, 4)); TRY(per_scan(eng, d.full_list, 1)); TRY(per_scan(eng, d.cf_tasks, d.cf_tiles));
    TRY(per_scan(eng, d.need2, 1)); TRY(per_scan(eng, d.far_arr, 1)); TRY(per_scan(eng, d.boxes, d.max_boxes));
    TRY(per_scan(eng, d.box_tests, d.max_boxes)); TRY(per_scan(eng, d.poses, 16)); TRY(per_scan(eng, d.occ_win, MW2 / 32));
    TRY(per_scan(eng, d.counts, d.n_classes)); TRY(per_scan(eng, d.cand_flags, K1)); TRY(per_scan(eng, d.cand_level, K1));
    TRY(per_scan(eng, d.cand_v, K1)); TRY(per_scan(eng, d.cand_list, K1)); TRY(per_scan(eng, d.n_list, 1));
    TRY(per_scan(eng, d.tickets, 4)); TRY(per_scan(eng, d.feas, d.K)); TRY(per_scan(eng, d.inserted, (size_t)d.max_events * 4));
    TRY(per_scan(eng, d.inserted_box, (size_t)d.max_events * 8)); TRY(per_scan(eng, d.check, (size_t)d.max_inserted * 5));
    TRY(per_scan(eng, d.out_count, 1)); TRY(per_scan(eng, d.gcell, GG)); TRY(per_scan(eng, d.gpts, d.max_points));
    TRY(per_scan(eng, d.gnear, GG)); TRY(per_scan(eng, d.gscratch, GG)); TRY(per_scan(eng, d.col_off, col_groups(d.cols) + 1));
    TRY(per_scan(eng, d.col_idx, d.max_points)); TRY(per_scan(eng, d.acell, GG)); TRY(per_scan(eng, d.apts, d.max_points));
    TRY(per_scan(eng, d.try_obj, 1)); TRY(per_scan(eng, d.chunk_cnt, d.max_chunks)); TRY(per_scan(eng, d.od_map_dims, 8));
    TRY(per_scan(eng, d.occ_far, OCC_FAR_CAP + 1));
    if (cfg->task == 1) TRY(per_scan(eng, d.occ_cnt, MW2));
    TRY(eng->active_count.alloc(R3D_MAX_SUB * 64 * 2)); TRY(eng->round_ctl.alloc(R3D_MAX_SUB * 32));
    TRY(eng->out_off.alloc(B + 1)); TRY(eng->check_off.alloc(B + 1)); TRY(eng->out_xyzi.alloc(B * P)); TRY(eng->out_label.alloc(B * P));
    TRY(eng->out_check.alloc(B * d.max_inserted * 5)); TRY(eng->n0_arr.alloc(B)); TRY(eng->nbox0_arr.alloc(B));
    TRY(eng->boxes0.alloc(B * d.max_boxes)); TRY(eng->cos_k.alloc(K1)); TRY(eng->sin_k.alloc(K1));
    TRY(eng->radii_sq.alloc(R3D_NUM_RADII)); TRY(eng->radii_ok.alloc(R3D_NUM_RADII)); TRY(eng->classes.alloc(R3D_MAX_CLASSES));
    TRY(eng->od_map_off.alloc(B * 2 + 1)); TRY(eng->stats.alloc(R3D_N_STATS));
    d.active_count = eng->active_count.p; d.out_off = eng->out_off.p; d.check_off = eng->check_off.p;
    d.out_xyzi = eng->out_xyzi.p; d.out_label = eng->out_label.p; d.out_check = eng->out_check.p;
    d.cos_k = eng->cos_k.p; d.sin_k = eng->sin_k.p; d.radii_sq = eng->radii_sq.p; d.radii_ok = eng->radii_ok.p;
    d.classes = eng->classes.p; d.od_map_off = eng->od_map_off.p; d.stats = eng->stats.p;
    R3D_CUDA(cudaMemset(d.work_cnt, 0, B * 4 * sizeof(int)));
    R3D_CUDA(cudaMemset(d.need2, 0, B * sizeof(int)));
    R3D_CUDA(cudaMemset(d.tickets, 0, B * 4 * sizeof(unsigned)));
    R3D_CUDA(cudaMemset(d.stats, 0, R3D_N_STATS * sizeof(unsigned long long)));
    R3D_CUDA(cudaMemset(d.occ_far, 0xFF, B * (OCC_FAR_CAP + 1) * sizeof(int)));
    R3D_CUDA(cudaHostAlloc((void**)&eng->h_words, R3D_MAX_SUB * 64 * sizeof(unsigned long long), cudaHostAllocMapped));
    memset(eng->h_words, 0, R3D_MAX_SUB * 64 * sizeof(unsigned long long));
    R3D_CUDA(cudaHostGetDevicePointer((void**)&eng->d_words, eng->h_words, 0));
    R3D_CUDA(cudaMallocHost((void**)&eng->h_offsets, (2 * (B + 1) + 1) * sizeof(long long)));
    R3D_CUDA(cudaMemcpy(eng->classes.p, cls.data(), cls.size() * sizeof(ClassCfg), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->radii_sq.p, cfg->radii_sq, sizeof(cfg->radii_sq), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->radii_ok.p, cfg->radii_ok, sizeof(cfg->radii_ok), cudaMemcpyHostToDevice));
    k_fill_u64<<<148 * 4, 256, 0, eng->stream>>>(d.obj_raw, B * d.hw, R3D_EMPTY_U64); r3d_count_launch();
    R3D_CUDA(cudaMemsetAsync(d.dmask, 0, B * d.dwords * sizeof(unsigned), eng->stream));
    R3D_CUDA(cudaStreamSynchronize(eng->stream));
    *out = owner.release();
    return R3D_OK;
}

extern "C" int r3d_engine_destroy(r3d_engine* eng) {
    if (!bind(eng)) return R3D_OK;
    cudaStreamSynchronize(eng->stream);
    drain_events(eng);
    delete eng;
    return R3D_OK;
}

extern "C" int r3d_engine_set_yaw_tables(r3d_engine* eng, const double* cos_k, const double* sin_k) {
    if (!bind(eng) || !cos_k || !sin_k) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_yaw_tables: null argument");
    const size_t n = (size_t)eng->dev.K + 1;
    R3D_CUDA(cudaMemcpy(eng->cos_k.p, cos_k, n * sizeof(double), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->sin_k.p, sin_k, n * sizeof(double), cudaMemcpyHostToDevice));
    eng->yaw_set = true;
    return R3D_OK;
}

extern "C" int r3d_engine_set_objects(r3d_engine* eng, const r3d_object_db* db) {
    if (!bind(eng) || !db || db->n_objects <= 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_objects: bad argument");
    EngineDev& d = eng->dev;
    const int n = db->n_objects;
    const int64_t total = db->point_offsets[n];
    std::vector<double> x(total), y(total), z(total);
    std::vector<float> in(total);
    std::vector<unsigned> lab(total);
    for (int64_t i = 0; i < total; ++i) {
        const double* p = db->points5 + i * 5;
        x[i] = p[0]; y[i] = p[1]; z[i] = p[2]; in[i] = (float)p[3]; lab[i] = (unsigned)p[4];
    }
    std::vector<ObjBox> ob(n);
    int max_pts = 1;
    for (int o = 0; o < n; ++o) {
        const double* bx = db->boxes + (size_t)o * 8;
        ObjBox& t = ob[o];
        t.cx = bx[0]; t.cy = bx[1]; t.cz = bx[2]; t.a = bx[3]; t.b = bx[4];
        t.length = bx[5]; t.width = bx[6]; t.height = bx[7];
        t.rho = std::hypot(t.cx, t.cy); t.psi0 = std::atan2(t.cy, t.cx);
        t.reach = 0.5 * std::hypot(t.length, t.width) + 0.05;
        t.cls = db->class_index[o];
        t.first = (int)db->point_offsets[o]; t.count = (int)(db->point_offsets[o + 1] - db->point_offsets[o]);
        t.pad = 0;
        t.eu0 = t.ev0 = t.ez0 = 1e300; t.eu1 = t.ev1 = t.ez1 = -1e300;
        for (int i = t.first; i < t.first + t.count; ++i) {
            const double dx = x[i] - t.cx, dy = y[i] - t.cy;
            const double u = dx * t.a + dy * t.b, v = -dx * t.b + dy * t.a, w = z[i] - t.cz;
            t.eu0 = std::min(t.eu0, u); t.eu1 = std::max(t.eu1, u); t.ev0 = std::min(t.ev0, v); t.ev1 = std::max(t.ev1, v);
            t.ez0 = std::min(t.ez0, w); t.ez1 = std::max(t.ez1, w);
        }
        t.eu0 -= 1e-6; t.ev0 -= 1e-6; t.ez0 -= 1e-6; t.eu1 += 1e-6; t.ev1 += 1e-6; t.ez1 += 1e-6;
        if (t.cls < 0 || t.cls >= d.n_classes) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_objects: class index out of range");
        max_pts = std::max(max_pts, t.count);
    }
    if (max_pts > 32768) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_set_objects: a cut object has more than 32768 points");
    d.max_obj_points = max_pts; d.n_objects = n;
    TRY(eng->obj_x.alloc(total)); TRY(eng->obj_y.alloc(total)); TRY(eng->obj_z.alloc(total)); TRY(eng->obj_i.alloc(total));
    TRY(eng->obj_label.alloc(total)); TRY(eng->obj.alloc(n)); TRY(eng->class_list_off.alloc(d.n_classes + 1));
    const int nl = db->class_list_offsets[d.n_classes];
    TRY(eng->class_list.alloc(std::max(nl, 1)));
    TRY(per_scan(eng, d.unplaceable, (n + 31) / 32));
    TRY(per_scan(eng, d.occ_pix, (size_t)OCC_G * max_pts)); TRY(per_scan(eng, d.sel_pix, max_pts));
    R3D_CUDA(cudaMemcpy(eng->obj_x.p, x.data(), total * sizeof(double), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->obj_y.p, y.data(), total * sizeof(double), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->obj_z.p, z.data(), total * sizeof(double), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->obj_i.p, in.data(), total * sizeof(float), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->obj_label.p, lab.data(), total * sizeof(unsigned), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->obj.p, ob.data(), n * sizeof(ObjBox), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->class_list_off.p, db->class_list_offsets, (d.n_classes + 1) * sizeof(int), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->class_list.p, db->class_list, nl * sizeof(int), cudaMemcpyHostToDevice));
    d.obj_x = eng->obj_x.p; d.obj_y = eng->obj_y.p; d.obj_z = eng->obj_z.p; d.obj_i = eng->obj_i.p; d.obj_label = eng->obj_label.p;
    d.obj = eng->obj.p; d.class_list_off = eng->class_list_off.p; d.class_list = eng->class_list.p;
    const size_t sel_smem = select_smem_bytes(std::min(max_pts, SEL_SMEM_PTS));
    d.sel_key_cap = next_pow2(max_pts);
    if (max_pts > std::min(SEL_SMEM_PTS, walk_od::WALK_SEL_PTS)) {        // objects the selection cannot keep in shared memory
        TRY(per_scan(eng, d.sel_keys, d.sel_key_cap)); TRY(per_scan(eng, d.sel_r, max_pts));
    }
    R3D_CUDA(cudaFuncSetAttribute(k_select_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sel_smem));
    R3D_CUDA(cudaFuncSetAttribute(k_occl_count, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)occl_smem_bytes(d)));
    if (onmap_smem_bytes(d.K) > 100 * 1024) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_set_objects: too many yaw steps for the placement kernel's shared memory");
    R3D_CUDA(cudaFuncSetAttribute(k_onmap, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)onmap_smem_bytes(d.K)));
    if (grid_near_smem(d.G) > 200 * 1024) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_set_objects: road-level grid too large for shared memory");
    R3D_CUDA(cudaFuncSetAttribute(k_grid_near_bits, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)grid_near_smem(d.G)));
    if (std::max(walk_od::walk_smem_layout(d.K, d.dwords).total, walk_ss::walk_smem_layout(d.K, d.dwords).total) > 200 * 1024)
        return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_set_objects: range image / yaw steps too large for the walker's shared memory");
    R3D_CUDA(cudaFuncSetAttribute(walk_od::k_scan_walk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)walk_od::walk_smem_layout(d.K, d.dwords).total));
    R3D_CUDA(cudaFuncSetAttribute(walk_ss::k_scan_walk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)walk_ss::walk_smem_layout(d.K, d.dwords).total));
    // the device schedule draw of r3d_engine_load_resident, which refuses a larger max_tries (the host path takes any)
    if (d.max_tries <= DRAW_MAX_TRIES) R3D_CUDA(allow_draw_schedule_smem(d.max_tries));
    eng->objects_set = true;
    return R3D_OK;
}

extern "C" int r3d_engine_set_ss_map(r3d_engine* eng, const uint8_t* map, int32_t size_x, int32_t size_y, int64_t move_x,
                                     int64_t move_y) {
    if (!bind(eng) || !map || size_x <= 0 || size_y <= 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_ss_map: bad argument");
    TRY(eng->ss_map.alloc((size_t)size_x * size_y));
    R3D_CUDA(cudaMemcpy(eng->ss_map.p, map, (size_t)size_x * size_y, cudaMemcpyHostToDevice));
    eng->dev.ss_map = eng->ss_map.p; eng->dev.ss_sx = size_x; eng->dev.ss_sy = size_y;
    eng->dev.ss_move_x = move_x; eng->dev.ss_move_y = move_y;
    return R3D_OK;
}

// per-box collision tests of the loaded batch's scene boxes
static void launch_box_tests(r3d_engine* eng) {
    const int slots = eng->n_scans * eng->dev.max_boxes;
    k_box_tests<<<(slots + 127) / 128, 128, 0, eng->stream>>>(eng->dev.boxes, eng->dev.box_tests, slots);
    r3d_count_launch();
}

// the scene boxes as loaded: drops the boxes appended by the previous run (device to device)
static int restore_scene_boxes(r3d_engine* eng) {
    const size_t slots = (size_t)eng->n_scans * eng->dev.max_boxes;
    R3D_CUDA(cudaMemcpyAsync(eng->dev.boxes, eng->boxes0.p, slots * sizeof(Box), cudaMemcpyDeviceToDevice, eng->stream));
    launch_box_tests(eng);
    return R3D_OK;
}

static int arm_batch(r3d_engine* eng, bool ingest) {
    eng->run_active = false;                     // a new batch / re-arm abandons a run that was left unfinished
    EngineDev& d = eng->dev;
    const int n = eng->n_scans;
    cudaStream_t st = eng->stream;
    k_reset_state<<<(n + 127) / 128, 128, 0, st>>>(d, n, eng->n0_arr.p, eng->nbox0_arr.p); r3d_count_launch();
    R3D_CUDA(cudaMemsetAsync(d.dmask, 0, (size_t)n * d.dwords * sizeof(unsigned), st));   // vis_px masks: cleared lazily afterwards
    const int chunks = (eng->max_n0 + CHUNK - 1) / CHUNK;
    if (ingest) {
        R3D_CUDA(cudaMemsetAsync(d.gcell, 0, (size_t)n * d.G * d.G * sizeof(int), st));
        R3D_CUDA(cudaMemsetAsync(d.col_off, 0, (size_t)n * (col_groups(d.cols) + 1) * sizeof(int), st));
        R3D_CUDA(cudaMemsetAsync(d.acell, 0, (size_t)n * d.G * d.G * sizeof(int), st));
        { Launcher l(eng, KID_INGEST); k_ingest_count<<<dim3(chunks, n), STREAM_THREADS, 0, st>>>(d, n); }
        {
            Launcher l(eng, KID_GRID);
            k_bucket_scan3<<<dim3(n, 3), 1024, 0, st>>>(d, n);
        }
        { Launcher l(eng, KID_SCATTER); k_scatter_project<<<dim3(chunks, n), STREAM_THREADS, 0, st>>>(d, n); }
        {
            Launcher l(eng, KID_GRID);
            k_grid_near_bits<<<n, NEAR_THREADS, grid_near_smem(d.G), st>>>(d, n);
        }
        eng->fresh = true;                       // the first range image of every scan is already projected
    } else {
        eng->fresh = false;
        k_reset_alive<<<dim3(std::max(chunks, 1), n), 256, 0, st>>>(d, n); r3d_count_launch();
        TRY(restore_scene_boxes(eng));
    }
    eng->ran = false;
    return r3d_check_launch("arm_batch");
}

// Checks that a batch fits the engine before anything of it is enqueued, and makes it the loaded shape: points[s]
// points and boxes[s] scene boxes in scan s, at most `objects` objects in any scan's schedule.  The errors name the
// entry point `fn`.
static int set_batch_shape(r3d_engine* eng, const char* fn, const std::vector<int64_t>& points, const std::vector<int>& boxes,
                           long long objects) {
    const EngineDev& d = eng->dev;
    auto fail = [fn](const char* what) { return r3d_fail(R3D_ERR_CAPACITY, (std::string(fn) + ": " + what).c_str()); };
    int max_n0 = 0;
    for (size_t s = 0; s < points.size(); ++s) {
        if (points[s] <= 0 || points[s] > d.max_points) return fail("scan larger than max_points (or empty)");
        if (boxes[s] > d.max_boxes) return fail("too many scene boxes");
        max_n0 = std::max(max_n0, (int)points[s]);
    }
    if (objects + 1 > d.max_events)                 // a schedule must fit the per-scan event / insertion records
        return fail("a scan's schedule asks for more objects than max_events - 1 "
                    "(create the engine with max_events = objects per scan + 1)");
    eng->n_scans = (int)points.size();
    eng->max_n0 = max_n0;
    eng->h_nbox0 = boxes;
    return R3D_OK;
}

extern "C" int r3d_engine_load_batch(r3d_engine* eng, const r3d_batch* bt) {
    if (!bind(eng) || !bt) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_batch: null argument");
    if (!eng->objects_set || !eng->yaw_set) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_batch: set objects and yaw tables first");
    EngineDev& d = eng->dev;
    const int n = bt->n_scans;
    if (n <= 0 || n > d.B) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_load_batch: n_scans exceeds max_scans");
    if (!bt->point_offsets || !bt->xyzi || (!bt->labels && !bt->labels16 && !bt->labels1) || !bt->counts || !bt->perms || bt->n_events <= 0)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_batch: missing arrays");
    if (d.task == 1 && (!bt->poses || !d.ss_map)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_batch: semseg needs poses and the map");
    if (d.task == 0 && (!bt->maps || !bt->map_offsets || !bt->map_dims)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_batch: OD needs maps");
    cudaStream_t st = eng->stream;
    std::vector<int64_t> points(n);
    std::vector<int> nb(n, 0);
    long long objects = 0;
    for (int s = 0; s < n; ++s) {
        points[s] = bt->point_offsets[s + 1] - bt->point_offsets[s];
        if (bt->box_offsets) nb[s] = bt->box_offsets[s + 1] - bt->box_offsets[s];
        long long want = 0;
        for (int c = 0; c < d.n_classes; ++c) want += std::max(bt->counts[(size_t)s * d.n_classes + c], 0);
        objects = std::max(objects, want);
    }
    TRY(set_batch_shape(eng, "r3d_engine_load_batch", points, nb, objects));
    const std::vector<int> n0(points.begin(), points.end());
    // scene boxes
    std::vector<Box> h_boxes((size_t)n * d.max_boxes);
    for (int s = 0; s < n; ++s)
        for (int j = 0; j < nb[s]; ++j) {
            const double* src = bt->boxes + ((size_t)bt->box_offsets[s] + j) * R3D_BOX_DOUBLES;
            Box& b = h_boxes[(size_t)s * d.max_boxes + j];
            b.cx = src[0]; b.cy = src[1]; b.cz = src[2];
            for (int i = 0; i < 9; ++i) b.m[i] = src[3 + i];
            b.length = src[12]; b.width = src[13]; b.height = src[14]; b.reach = src[15];
        }
    R3D_CUDA(cudaMemcpyAsync(d.boxes, h_boxes.data(), h_boxes.size() * sizeof(Box), cudaMemcpyHostToDevice, st));
    R3D_CUDA(cudaMemcpyAsync(eng->boxes0.p, d.boxes, h_boxes.size() * sizeof(Box), cudaMemcpyDeviceToDevice, st));
    launch_box_tests(eng);
    R3D_CUDA(cudaMemcpyAsync(eng->n0_arr.p, n0.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    R3D_CUDA(cudaMemcpyAsync(eng->nbox0_arr.p, nb.data(), n * sizeof(int), cudaMemcpyHostToDevice, st));
    if (d.task == 0) {
        const int64_t bytes = bt->map_offsets[(size_t)n * 2];
        if ((size_t)bytes > eng->od_maps.n) TRY(eng->od_maps.alloc((size_t)bytes));
        R3D_CUDA(cudaMemcpyAsync(eng->od_maps.p, bt->maps, (size_t)bytes, cudaMemcpyHostToDevice, st));
        R3D_CUDA(cudaMemcpyAsync(eng->od_map_off.p, bt->map_offsets, ((size_t)n * 2 + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
        R3D_CUDA(cudaMemcpyAsync(mut(d.od_map_dims), bt->map_dims, (size_t)n * 8 * sizeof(int), cudaMemcpyHostToDevice, st));
        d.od_maps = eng->od_maps.p;
    } else {
        R3D_CUDA(cudaMemcpyAsync(mut(d.poses), bt->poses, (size_t)n * 16 * sizeof(double), cudaMemcpyHostToDevice, st));
    }
    R3D_CUDA(cudaMemcpyAsync(mut(d.counts), bt->counts, (size_t)n * d.n_classes * sizeof(int), cudaMemcpyHostToDevice, st));
    const size_t nperm = (size_t)n * bt->n_events * d.n_classes * d.max_tries;
    if (nperm > eng->perms.n) TRY(eng->perms.alloc(nperm));
    R3D_CUDA(cudaMemcpyAsync(eng->perms.p, bt->perms, nperm * sizeof(int), cudaMemcpyHostToDevice, st));
    d.perms = eng->perms.p; d.n_perm_events = bt->n_events;
    // points: packed host rows -> per-scan strided device rows (one pitched copy when every scan has the same size)
    bool uniform = true;
    for (int s = 1; s < n; ++s) uniform &= n0[s] == n0[0];
    const bool packed = bt->labels == nullptr;         // 16-bit labels / Road bits: staged contiguously, expanded on the device
    const bool bits = packed && bt->labels16 == nullptr;
    if (bits && (d.task != 0 || bt->point_offsets[0] != 0))
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_batch: labels1 (one Road bit per point) is for object detection batches that start at point 0");
    if (packed) {
        const size_t total = (size_t)(bt->point_offsets[n] - bt->point_offsets[0]);
        if ((size_t)n + 1 > eng->pt_off.n) TRY(eng->pt_off.alloc((size_t)d.B + 1));
        if (bits) {
            const size_t nbytes = (total + 7) / 8;
            if (nbytes > eng->label1.n) TRY(eng->label1.alloc(nbytes));
            R3D_CUDA(cudaMemcpyAsync(eng->label1.p, bt->labels1, nbytes, cudaMemcpyHostToDevice, st));
        } else {
            if (total > eng->label16.n) TRY(eng->label16.alloc(total));
            R3D_CUDA(cudaMemcpyAsync(eng->label16.p, bt->labels16 + bt->point_offsets[0], total * sizeof(unsigned short), cudaMemcpyHostToDevice, st));
        }
        R3D_CUDA(cudaMemcpyAsync(eng->pt_off.p, bt->point_offsets, ((size_t)n + 1) * sizeof(long long), cudaMemcpyHostToDevice, st));
    }
    if (uniform) {
        R3D_CUDA(cudaMemcpy2DAsync(mut(d.xyzi), (size_t)d.max_points * sizeof(float4), bt->xyzi + bt->point_offsets[0] * 4,
                                   (size_t)n0[0] * sizeof(float4), (size_t)n0[0] * sizeof(float4), n, cudaMemcpyHostToDevice, st));
        if (!packed)
            R3D_CUDA(cudaMemcpy2DAsync(d.label, (size_t)d.P * sizeof(unsigned), bt->labels + bt->point_offsets[0],
                                       (size_t)n0[0] * sizeof(unsigned), (size_t)n0[0] * sizeof(unsigned), n, cudaMemcpyHostToDevice, st));
    } else {
        for (int s = 0; s < n; ++s) {
            const int64_t o = bt->point_offsets[s];
            R3D_CUDA(cudaMemcpyAsync(mut(d.xyzi) + (size_t)s * d.max_points, bt->xyzi + o * 4, (size_t)n0[s] * sizeof(float4), cudaMemcpyHostToDevice, st));
            if (!packed)
                R3D_CUDA(cudaMemcpyAsync(d.label + (size_t)s * d.P, bt->labels + o, (size_t)n0[s] * sizeof(unsigned), cudaMemcpyHostToDevice, st));
        }
    }
    if (packed) {
        const int chunks = (eng->max_n0 + CHUNK - 1) / CHUNK;
        if (bits) k_expand_label_bits<<<dim3(chunks, n), STREAM_THREADS, 0, st>>>(eng->label1.p, eng->pt_off.p, d.label, d.P, n, (unsigned)d.road_label);
        else k_widen_labels<<<dim3(chunks, n), STREAM_THREADS, 0, st>>>(eng->label16.p, eng->pt_off.p, d.label, d.P, n);
        r3d_count_launch();
    }
    // the std::vectors above are pageable: the copies from them completed before cudaMemcpyAsync returned
    eng->batch_loaded = true;
    eng->from_store = false;                         // host batches are never world-augmented
    eng->world_loaded = false;
    d.world = nullptr;
    return arm_batch(eng, true);
}

extern "C" int r3d_engine_set_schedule_policy(r3d_engine* eng, int32_t random, int32_t number_of_object, const int32_t* fixed_counts) {
    if (!bind(eng) || (random && number_of_object < 0) || (!random && !fixed_counts))
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_schedule_policy: bad argument");
    SchedulePolicy p;
    memset(&p, 0, sizeof(p));
    p.random = random ? 1 : 0;
    p.number_of_object = random ? number_of_object : 0;
    for (int c = 0; !random && c < eng->dev.n_classes; ++c) {
        if (fixed_counts[c] < 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_schedule_policy: negative class count");
        p.fixed[c] = fixed_counts[c];
    }
    eng->policy = p;
    eng->policy_set = true;
    return R3D_OK;
}

extern "C" int r3d_engine_load_resident(r3d_engine* eng, const r3d_resident_store* s, const int32_t* indices, int32_t n,
                                        uint64_t seed, uint64_t epoch) {
    if (!bind(eng) || !s || !indices) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_resident: null argument");
    if (!eng->objects_set || !eng->yaw_set) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_resident: set objects and yaw tables first");
    if (!eng->policy_set) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_resident: set the schedule policy first");
    EngineDev& d = eng->dev;
    if (d.max_tries > DRAW_MAX_TRIES)
        return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_load_resident: max_tries above 4266, the most the device schedule draw takes");
    if (n <= 0 || n > d.B) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_load_resident: n_scans exceeds max_scans");
    if (s->n_scans <= 0 || !s->xyzi || ((uintptr_t)s->xyzi & 15) || !s->labels || !s->point_offsets || !s->box_offsets ||
        !s->h_point_offsets || !s->h_box_offsets || (!s->boxes && s->h_box_offsets[s->n_scans] > 0))
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_resident: missing store arrays");
    if (d.task == 1 && (!s->poses || !d.ss_map)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_resident: semseg needs poses and the map");
    if (d.task == 0 && (!s->maps || !s->map_offsets || !s->map_dims)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_resident: OD needs maps");
    // the checks of r3d_engine_load_batch, on the host copies of the store's offsets
    std::vector<int64_t> points(n);
    std::vector<int> nb(n);
    for (int b = 0; b < n; ++b) {
        const int i = indices[b];
        if (i < 0 || i >= s->n_scans) return r3d_fail(R3D_ERR_ARG, "r3d_engine_load_resident: index out of range");
        points[b] = s->h_point_offsets[i + 1] - s->h_point_offsets[i];
        nb[b] = s->h_box_offsets[i + 1] - s->h_box_offsets[i];
    }
    long long objects = eng->policy.number_of_object;
    if (!eng->policy.random) { objects = 0; for (int c = 0; c < d.n_classes; ++c) objects += eng->policy.fixed[c]; }
    TRY(set_batch_shape(eng, "r3d_engine_load_resident", points, nb, objects));
    const size_t nperm = (size_t)d.B * d.max_events * d.n_classes * d.max_tries;
    if (nperm > eng->perms.n) TRY(eng->perms.alloc(nperm));
    if (!eng->h_idx) {
        R3D_CUDA(cudaMallocHost((void**)&eng->h_idx, (size_t)d.B * sizeof(int)));
        R3D_CUDA(cudaEventCreateWithFlags(&eng->ev_idx, cudaEventDisableTiming));
        TRY(eng->idx_dev.alloc(d.B));
    }
    if (eng->world_on && !eng->world.p) TRY(eng->world.alloc((size_t)d.B * 8));
    cudaStream_t st = eng->stream;
    R3D_CUDA(cudaEventSynchronize(eng->ev_idx));
    memcpy(eng->h_idx, indices, (size_t)n * sizeof(int));
    R3D_CUDA(cudaMemcpyAsync(eng->idx_dev.p, eng->h_idx, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, st));
    R3D_CUDA(cudaEventRecord(eng->ev_idx, st));
    const int* idx = eng->idx_dev.p;
    const int od = d.task == 0;
    launch_gather_points(*s, idx, n, eng->max_n0, mut(d.xyzi), d.max_points, d.label, d.P, od, (unsigned)d.road_label, st);
    launch_gather_meta(*s, idx, n, od, eng->n0_arr.p, eng->nbox0_arr.p, eng->od_map_off.p, mut(d.od_map_dims), mut(d.poses),
                       d.boxes, eng->boxes0.p, d.max_boxes, st);
    launch_box_tests(eng);
    if (od) d.od_maps = s->maps;
    d.perms = eng->perms.p; d.n_perm_events = d.max_events;
    launch_draw_schedule(idx, n, d.max_events, d.n_classes, d.max_tries, d.class_list_off, eng->policy, seed, epoch, mut(d.counts),
                         eng->perms.p, st);
    if (eng->world_on) launch_draw_world(idx, n, eng->world_pol, seed, epoch, eng->world.p, st);
    d.world = eng->world_on ? eng->world.p : nullptr;
    eng->world_loaded = eng->world_on;
    eng->from_store = true;
    eng->targets_bound = 0;
    eng->batch_idx.assign(indices, indices + n);
    TRY(r3d_check_launch("r3d_engine_load_resident"));
    eng->batch_loaded = true;
    return arm_batch(eng, true);
}

extern "C" int r3d_engine_set_ss_map_device(r3d_engine* eng, const uint8_t* map, int32_t size_x, int32_t size_y, int64_t move_x,
                                            int64_t move_y) {
    if (!bind(eng) || !map || size_x <= 0 || size_y <= 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_ss_map_device: bad argument");
    eng->dev.ss_map = map; eng->dev.ss_sx = size_x; eng->dev.ss_sy = size_y;
    eng->dev.ss_move_x = move_x; eng->dev.ss_move_y = move_y;
    return R3D_OK;
}

extern "C" int r3d_engine_schedule_read(r3d_engine* eng, int32_t* counts, int32_t* perms, int32_t* n_events) {
    if (!bind(eng) || !counts || !n_events || !eng->batch_loaded) return r3d_fail(R3D_ERR_ARG, "r3d_engine_schedule_read: bad argument or no batch");
    const EngineDev& d = eng->dev;
    R3D_CUDA(engine_wait(eng));
    const size_t n = (size_t)eng->n_scans;
    R3D_CUDA(cudaMemcpy(counts, d.counts, n * d.n_classes * sizeof(int), cudaMemcpyDeviceToHost));
    if (perms) R3D_CUDA(cudaMemcpy(perms, d.perms, n * d.n_perm_events * d.n_classes * d.max_tries * sizeof(int), cudaMemcpyDeviceToHost));
    *n_events = d.n_perm_events;
    return R3D_OK;
}

extern "C" int r3d_engine_reset_batch(r3d_engine* eng) {
    if (!bind(eng) || !eng->batch_loaded) return r3d_fail(R3D_ERR_ARG, "r3d_engine_reset_batch: no batch loaded");
    return arm_batch(eng, false);
}

extern "C" int r3d_engine_rearm_batch(r3d_engine* eng, int from_raw_points) {
    if (!bind(eng) || !eng->batch_loaded) return r3d_fail(R3D_ERR_ARG, "r3d_engine_rearm_batch: no batch loaded");
    if (!from_raw_points) return arm_batch(eng, false);
    // the whole device path from the resident float4 points again: scene boxes, spherical ingest, spatial indices
    TRY(restore_scene_boxes(eng));
    return arm_batch(eng, true);
}

// view of the device data model that starts at scan b0: every per-scan array is [scan][...], so offsetting the base
// pointers lets the kernels run unchanged on a contiguous sub-batch
static EngineDev sub_view(const r3d_engine* eng, int b0) {
    EngineDev v = eng->dev;
    if (b0 == 0) return v;
    char* base = reinterpret_cast<char*>(&v);
    for (const r3d_engine::PerScan& a : eng->scan_arrays) {
        char* p;
        memcpy(&p, base + a.field, sizeof(p));
        p += (size_t)b0 * a.stride;
        memcpy(base + a.field, &p, sizeof(p));
    }
    // perms: [n][n_perm_events][C][tries] of the loaded schedule, not of its allocation; od_map_off: [B][2] + an end slot
    if (v.perms) v.perms += (size_t)b0 * v.n_perm_events * v.n_classes * v.max_tries;
    if (v.od_map_off) v.od_map_off += (size_t)b0 * 2;
    return v;
}

extern "C" int r3d_engine_run_until(r3d_engine* eng, int stop_at, int* still_running);

extern "C" int r3d_engine_run(r3d_engine* eng) { return r3d_engine_run_until(eng, 0, nullptr); }

// output compaction of the batch after its last round, and the read-back of the point / check row offsets
static int launch_output(r3d_engine* eng, int chunks_all) {
    const EngineDev& d = eng->dev;
    const int n = eng->n_scans;
    cudaStream_t st = eng->stream;
    {
        Launcher l(eng, KID_OUT);
        k_out_count<<<dim3(chunks_all, n), STREAM_THREADS, 0, st>>>(d, n);
        k_out_offsets<<<1, 1024, 0, st>>>(d, n, chunks_all);
        if (d.world) k_out_write<true><<<dim3(chunks_all, n), STREAM_THREADS, 0, st>>>(d, n);
        else k_out_write<false><<<dim3(chunks_all, n), STREAM_THREADS, 0, st>>>(d, n);
        r3d_count_launch(2);
    }
    R3D_CUDA(cudaMemcpyAsync(eng->h_offsets, eng->out_off.p, (n + 1) * sizeof(long long), cudaMemcpyDeviceToHost, st));
    R3D_CUDA(cudaMemcpyAsync(eng->h_offsets + (d.B + 1), eng->check_off.p, (n + 1) * sizeof(long long), cudaMemcpyDeviceToHost, st));
    eng->ran = true;
    return R3D_OK;
}

// The default execution model: batch-wide streaming kernels for the first range image of every scan, then ONE launch
// of the per-scan walker (r3d_k_walk.cuh) that takes every scan through all its slots and tries, then the output
// compaction.  Everything is queued on the engine stream; the host neither polls nor synchronises.
static int run_walker(r3d_engine* eng) {
    const EngineDev& d = eng->dev;
    const int n = eng->n_scans;
    cudaStream_t st = eng->stream;
    const int chunks0 = (eng->max_n0 + CHUNK - 1) / CHUNK;
    const int chunks_all = (eng->max_n0 + d.max_inserted + CHUNK - 1) / CHUNK;
    const int full_y = std::min(n, R3D_FULL_Y);
    const bool fresh = eng->fresh;
    eng->fresh = false;
    { Launcher l(eng, KID_PREP); walk_od::k_walk_prepare<<<std::min((n * d.cf_tiles + 255) / 256, eng->n_sms * 4), 256, 0, st>>>(d, n, fresh ? 0 : 1); }
    if (!fresh) {                                // re-armed without ingest: rebuild the first range image from the caches
        { Launcher l(eng, KID_MINMAX0); k_minmax<<<dim3(chunks0, full_y), STREAM_THREADS, 0, st>>>(d, n); }
        { Launcher l(eng, KID_CLEAR0); k_clear_images<<<dim3(32, full_y), STREAM_THREADS, 0, st>>>(d, n); }
        { Launcher l(eng, KID_PROJECT0); k_project<<<dim3(chunks0, full_y), STREAM_THREADS, 0, st>>>(d, n); }
    }
    {
        Launcher l(eng, KID_CLOSEFILL0);
        const int cf_grid = std::min(n * d.cf_tiles, eng->n_sms * 4);
        if (eng->zraw_tmap_ok) {                 // tile loads by the TMA unit
            k_close_fill_tma<<<cf_grid, CF_THREADS, 0, st>>>(eng->zraw_tmap, d.rows, d.cols, (int64_t)d.hw, d.smooth, d.far_arr, d.cf_tasks,
                                                              d.work_cnt + 1);
        } else if ((d.cols & 1) == 0 && ((uintptr_t)d.zraw & 15) == 0) {
            k_close_fill_raw_pipelined<<<cf_grid, CF_THREADS, 0, st>>>(d.zraw, d.rows, d.cols, (int64_t)d.hw, d.smooth, d.far_arr, d.cf_tasks,
                                                                        d.work_cnt + 1);
        } else {
            RawImage in{d.zraw};
            k_close_fill_tasks<RawImage><<<cf_grid, CF_THREADS, 0, st>>>(in, d.rows, d.cols, (int64_t)d.hw, d.smooth, d.far_arr, d.cf_tasks,
                                                                         d.work_cnt + 1);
        }
    }
    if (d.task == 1) {
        R3D_CUDA(cudaMemsetAsync(d.occ_win, 0, (size_t)n * ((size_t)d.map_window * d.map_window / 32) * sizeof(unsigned), st));
        R3D_CUDA(cudaMemsetAsync(d.occ_cnt, 0, (size_t)n * (size_t)d.map_window * d.map_window * sizeof(unsigned), st));
        Launcher l(eng, KID_ADJUST); k_adjust_map<<<dim3(chunks0, n), STREAM_THREADS, 0, st>>>(d, n, 1);
    }
    {
        Launcher l(eng, KID_WALK);               // CTA shape per task: see the head of r3d_k_walk.cuh
        if (d.task == 1) walk_ss::k_scan_walk<<<n, walk_ss::WALK_THREADS, walk_ss::walk_smem_layout(d.K, d.dwords).total, st>>>(d, n);
        else walk_od::k_scan_walk<<<n, walk_od::WALK_THREADS, walk_od::walk_smem_layout(d.K, d.dwords).total, st>>>(d, n);
    }
    TRY(launch_output(eng, chunks_all));
    R3D_CUDA(cudaMemcpyAsync(eng->h_offsets + 2 * (d.B + 1), eng->stats.p + 8, sizeof(long long), cudaMemcpyDeviceToHost, st));
    eng->walked = true;
    return r3d_check_launch("r3d_engine_run");
}

extern "C" int r3d_engine_run_until(r3d_engine* eng, int stop_at, int* still_running) {
    if (!bind(eng) || !eng->batch_loaded) return r3d_fail(R3D_ERR_ARG, "r3d_engine_run: no batch loaded");
    if (still_running) *still_running = 0;
    if (!eng->staged) return run_walker(eng);
    eng->walked = false;
    const EngineDev& d0 = eng->dev;
    const int n = eng->n_scans;
    cudaStream_t st = eng->stream;
    const int P_live = eng->max_n0 + d0.max_inserted;
    const int chunks_all = (P_live + CHUNK - 1) / CHUNK;
    const int sel_pts = std::min(d0.max_obj_points, SEL_SMEM_PTS);
    const size_t sel_smem = select_smem_bytes(sel_pts);
    const int key_cap = next_pow2(sel_pts);
    const size_t onmap_smem = onmap_smem_bytes(d0.K);
    const int max_rounds = d0.max_events * (3 * d0.max_tries + 2) + 8;
    // The batch is advanced as n_sub contiguous sub-batches, each on its own stream: every kernel of a round is a
    // short chain of dependent loads that leaves most of the SMs' issue slots idle, so the rounds of different
    // sub-batches overlap on the device.
    typedef r3d_engine::Sub Sub;
    Sub* sub = eng->sub;
    if (!eng->run_active) {
        eng->run_nsub = std::max(1, std::min(eng->n_sub, n));
        eng->run_done = 0; eng->run_rounds = 0;
        R3D_CUDA(cudaEventRecord(eng->ev_armed, st));
        for (int i = 0; i < eng->run_nsub; ++i) {
            Sub& s = sub[i];
            s.b0 = (int)((long long)n * i / eng->run_nsub); s.n = (int)((long long)n * (i + 1) / eng->run_nsub) - s.b0;
            s.round = 0; s.done = false; s.left = s.n; s.d = sub_view(eng, s.b0); s.st = eng->sub_stream[i];
            s.d.active_count = eng->active_count.p + (size_t)i * 128;
            s.d.host_word = eng->d_words + (size_t)i * 64;
            s.d.round_ctl = eng->round_ctl.p + (size_t)i * 32;
            if (eng->seq > 0xF0000000u) eng->seq = 0;                       // sequence numbers are never 0 (= a fresh word)
            s.seq_base = eng->seq + 1; eng->seq += (unsigned)max_rounds + 8u;
            R3D_CUDA(cudaStreamWaitEvent(s.st, eng->ev_armed, 0));
            R3D_CUDA(cudaMemsetAsync(s.d.active_count, 0, 128 * sizeof(int), s.st));
            k_set_round<<<1, 1, 0, s.st>>>(s.d.round_ctl, s.seq_base); r3d_count_launch();
        }
        eng->run_active = true;
    }
    const int nsub = eng->run_nsub;
    int& n_done = eng->run_done;
    int& rounds_max = eng->run_rounds;
    const int task_ctas = std::max(eng->n_sms, eng->n_sms * TASK_CTAS_PER_SM / nsub);
    // The k_ctrl of every round publishes (sequence number, unfinished scans) into mapped host memory.  The host keeps
    // up to `ahead` rounds of a sub-batch in flight: round r is launched once the word of round r - ahead is there
    // (rounds launched after the last scan finished are gated off on the device and cost a few microseconds each),
    // so neither the device nor the other sub-batches ever wait for a word that is stuck behind bulk PCIe traffic.
    const int ahead = 3;
    auto poll_round = [&](int i, int round, long long& left) -> int {       // 1: published, 0: not yet
        volatile unsigned long long* w = eng->h_words + (size_t)i * 64 + (round & 63);
        const unsigned long long v = *w;
        if ((unsigned)(v >> 32) == sub[i].seq_base + (unsigned)round) { left = (long long)(v & 0xffffffffull); return 1; }
        return 0;
    };
    // the launch sequence of one round; also what a round graph is captured from
    auto launch_round = [&](const EngineDev& d, int ns, cudaStream_t ss, bool r0) {
        const size_t pref_smem = (size_t)(ns + 1) * sizeof(int);
        const int full_y = std::min(ns, R3D_FULL_Y);
        const int cf_grid = std::min(ns * d.cf_tiles, eng->n_sms * 8);
        { Launcher l(eng, KID_CTRL, ss); k_ctrl<<<ns, 32, 0, ss>>>(d, ns); }
        { Launcher l(eng, KID_UPDATE, ss); k_update<<<dim3(UPDATE_G, ns), UPDATE_THREADS, 0, ss>>>(d, ns); }
        { Launcher l(eng, r0 ? KID_MINMAX0 : KID_MINMAX, ss); k_minmax<<<dim3(chunks_all, full_y), STREAM_THREADS, 0, ss>>>(d, ns); }
        { Launcher l(eng, r0 ? KID_CLEAR0 : KID_CLEAR, ss); k_clear_images<<<dim3(32, full_y), STREAM_THREADS, 0, ss>>>(d, ns); }
        { Launcher l(eng, r0 ? KID_PROJECT0 : KID_PROJECT, ss); k_project<<<dim3(chunks_all, full_y), STREAM_THREADS, 0, ss>>>(d, ns); }
        {
            Launcher l(eng, r0 ? KID_CLOSEFILL0 : KID_CLOSEFILL, ss);
            if ((d.cols & 1) == 0 && ((uintptr_t)d.zraw & 15) == 0) {
                k_close_fill_raw_pipelined<<<std::min(cf_grid, eng->n_sms * 4), CF_THREADS, 0, ss>>>(d.zraw, d.rows, d.cols, (int64_t)d.hw, d.smooth, d.far_arr,
                                                                           d.cf_tasks, d.work_cnt + 1);
            } else {
                RawImage in{d.zraw};
                k_close_fill_tasks<RawImage><<<cf_grid, CF_THREADS, 0, ss>>>(in, d.rows, d.cols, (int64_t)d.hw, d.smooth, d.far_arr,
                                                                             d.cf_tasks, d.work_cnt + 1);
            }
        }
        if (d.task == 1) { Launcher l(eng, KID_ADJUST, ss); k_adjust_map<<<dim3(chunks_all, ns), STREAM_THREADS, 0, ss>>>(d, ns); }
        { Launcher l(eng, KID_ONMAP, ss); k_onmap<<<ns, TRY_THREADS, onmap_smem, ss>>>(d, ns); }
        const int ph = d.cand_window > 0 ? 1 : 0;           // OD: first window of candidates, then the rest where needed
        if (d.task == 0) { Launcher l(eng, KID_ONMAP, ss); k_onmap_full<<<task_ctas, TASK_THREADS, pref_smem, ss>>>(d, ns, ph); }
        { Launcher l(eng, KID_HEIGHT, ss); k_road_level<<<task_ctas, TASK_THREADS, pref_smem, ss>>>(d, ns, ph); }
        if (d.task == 1) {
            Launcher l(eng, KID_ONMAP, ss);
            if (d.K <= SS_MAX_K) k_onmap_ss<<<ns, 1024, 0, ss>>>(d, ns); else k_onmap_ss_seq<<<ns, 1024, 0, ss>>>(d, ns);
        }
        { Launcher l(eng, KID_COLLIDE, ss); k_collide<<<task_ctas, TASK_THREADS, pref_smem, ss>>>(d, ns, ph); }
        { Launcher l(eng, KID_OCCL, ss); k_occl_count<<<dim3(OCC_G, ns), 128, occl_smem_bytes(d), ss>>>(d, ns, ph); }
        if (ph) {
            { Launcher l(eng, KID_CTRL, ss); k_phase_gate<<<(ns + 127) / 128, 128, 0, ss>>>(d, ns); }
            { Launcher l(eng, KID_ONMAP, ss); k_onmap_full<<<task_ctas, TASK_THREADS, pref_smem, ss>>>(d, ns, 2); }
            { Launcher l(eng, KID_HEIGHT, ss); k_road_level<<<task_ctas, TASK_THREADS, pref_smem, ss>>>(d, ns, 2); }
            { Launcher l(eng, KID_COLLIDE, ss); k_collide<<<task_ctas, TASK_THREADS, pref_smem, ss>>>(d, ns, 2); }
            { Launcher l(eng, KID_OCCL, ss); k_occl_count<<<dim3(OCC_G, ns), 128, occl_smem_bytes(d), ss>>>(d, ns, 2); }
        }
        { Launcher l(eng, KID_SELECT, ss); k_select_emit<<<ns, 512, sel_smem, ss>>>(d, ns, key_cap, sel_pts); }
    };
    const bool graphs = eng->use_graphs && !eng->profile;
    if (graphs) {
        for (int i = 0; i < nsub; ++i) {
            r3d_engine::RoundGraph& g = eng->round_graph[i];
            const Sub& s = sub[i];
            if (g.exec && g.ns == s.n && g.chunks_all == chunks_all && g.task_ctas == task_ctas && g.sel_pts == sel_pts &&
                memcmp(&g.d, &s.d, sizeof(EngineDev)) == 0) continue;
            if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
            cudaGraph_t graph = nullptr;
            R3D_CUDA(cudaStreamBeginCapture(s.st, cudaStreamCaptureModeThreadLocal));
            eng->capturing = true;
            launch_round(s.d, s.n, s.st, false);
            eng->capturing = false;
            R3D_CUDA(cudaStreamEndCapture(s.st, &graph));
            size_t n_nodes = 0;
            R3D_CUDA(cudaGraphGetNodes(graph, nullptr, &n_nodes));
            const cudaError_t ie = cudaGraphInstantiate(&g.exec, graph, 0);
            cudaGraphDestroy(graph);
            if (ie != cudaSuccess) { g.exec = nullptr; return r3d_fail_cuda(ie, "r3d_engine_run: cudaGraphInstantiate"); }
            memcpy(&g.d, &s.d, sizeof(EngineDev));
            g.ns = s.n; g.chunks_all = chunks_all; g.task_ctas = task_ctas; g.sel_pts = sel_pts; g.kernels = (int)n_nodes;
        }
    }
    unsigned idle_polls = 0;
    while (n_done < nsub) {
        bool progressed = false;
        for (int i = 0; i < nsub; ++i) {
            Sub& s = sub[i];
            if (s.done) continue;
            if (s.round >= ahead) {                   // the word of round (s.round - ahead) gates the next launch
                long long left = 0;
                const int got = poll_round(i, s.round - ahead, left);
                if (got == 0) continue;
                s.left = left;
                if (left == 0) { s.done = true; ++n_done; progressed = true; rounds_max = std::max(rounds_max, s.round - ahead + 1); continue; }
            }
            progressed = true;
            if (s.round >= max_rounds) { eng->run_active = false; return r3d_fail(R3D_ERR_ARG, "r3d_engine_run: round limit reached"); }
            if (graphs) {
                R3D_CUDA(cudaGraphLaunch(eng->round_graph[i].exec, s.st));
                r3d_count_launch(eng->round_graph[i].kernels);
            } else {
                launch_round(s.d, s.n, s.st, s.round == 0);
            }
            s.round += 1;
        }
        if (stop_at > 0 && n_done < nsub) {             // hand the device to the next engine once only a tail is left
            long long left_total = 0;
            for (int i = 0; i < nsub; ++i) left_total += sub[i].done ? 0 : sub[i].left;
            if (left_total <= stop_at) { if (still_running) *still_running = 1; return R3D_OK; }
        }
        if (progressed) { idle_polls = 0; continue; }
        // nothing to launch: every unfinished sub-batch waits for a word.  Poll briefly, then sleep in short steps
        // instead of burning a host core per engine thread (8 ranks x 3 pipelined engines share the box's cores)
        if (++idle_polls > 64) std::this_thread::sleep_for(std::chrono::microseconds(20));
        if ((idle_polls & 0x3ff) == 0x3ff) {
            for (int i = 0; i < nsub; ++i) {
                if (sub[i].done) continue;
                const cudaError_t q = cudaStreamQuery(sub[i].st);
                long long left = 0;
                if ((q != cudaSuccess && q != cudaErrorNotReady) ||
                    (q == cudaSuccess && poll_round(i, sub[i].round - ahead, left) == 0))        // drained without the word
                    { eng->run_active = false; return r3d_fail_cuda(q == cudaSuccess ? cudaErrorUnknown : q, "r3d_engine_run: device error while waiting for a round"); }
            }
        }
    }
    eng->last_rounds = rounds_max;
    eng->run_active = false;
    for (int i = 0; i < nsub; ++i) {
        R3D_CUDA(cudaEventRecord(eng->sub_done[i], sub[i].st));
        R3D_CUDA(cudaStreamWaitEvent(st, eng->sub_done[i], 0));
    }
    TRY(launch_output(eng, chunks_all));
    return r3d_check_launch("r3d_engine_run");
}

extern "C" int r3d_engine_set_sub_batches(r3d_engine* eng, int n_sub) {
    if (!bind(eng) || n_sub < 1 || n_sub > R3D_MAX_SUB) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_sub_batches: 1..16");
    eng->n_sub = n_sub;
    return R3D_OK;
}

extern "C" int r3d_engine_sync(r3d_engine* eng) {
    if (!bind(eng)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_sync: null engine");
    R3D_CUDA(engine_wait(eng));
    drain_events(eng);
    return R3D_OK;
}

extern "C" int r3d_engine_output_rows(r3d_engine* eng, int64_t* total_points, int64_t* total_check) {
    if (!bind(eng) || !eng->ran) return r3d_fail(R3D_ERR_ARG, "r3d_engine_output_rows: run first");
    R3D_CUDA(engine_wait(eng));
    if (total_points) *total_points = eng->h_offsets[eng->n_scans];
    if (total_check) *total_check = eng->h_offsets[eng->dev.B + 1 + eng->n_scans];
    return R3D_OK;
}

extern "C" int r3d_engine_output_device(r3d_engine* eng, const float** out_xyzi, const uint32_t** out_labels, const float** check,
                                        int64_t* out_offsets_host, int64_t* check_offsets_host) {
    if (!bind(eng) || !eng->ran) return r3d_fail(R3D_ERR_ARG, "r3d_engine_output_device: run first");
    R3D_CUDA(engine_wait(eng));
    const int n = eng->n_scans;
    if (out_xyzi) *out_xyzi = reinterpret_cast<const float*>(eng->out_xyzi.p);
    if (out_labels) *out_labels = eng->out_label.p;
    if (check) *check = eng->out_check.p;
    if (out_offsets_host) memcpy(out_offsets_host, eng->h_offsets, (n + 1) * sizeof(long long));
    if (check_offsets_host) memcpy(check_offsets_host, eng->h_offsets + eng->dev.B + 1, (n + 1) * sizeof(long long));
    return R3D_OK;
}

extern "C" int r3d_engine_inserted_device(r3d_engine* eng, const int32_t** n_inserted, const int32_t** inserted,
                                          const double** inserted_box, const float** box7) {
    if (!bind(eng) || !eng->ran) return r3d_fail(R3D_ERR_ARG, "r3d_engine_inserted_device: run first");
    const EngineDev& d = eng->dev;
    if (!eng->n_ins_dev.p) { TRY(eng->n_ins_dev.alloc(d.B)); TRY(eng->box7.alloc((size_t)d.B * d.max_events * 7)); }
    launch_inserted_targets(eng->dev.st, eng->dev.inserted_box, eng->n_scans, d.max_events, eng->n_ins_dev.p, eng->box7.p, eng->stream);
    if (n_inserted) *n_inserted = eng->n_ins_dev.p;
    if (inserted) *inserted = eng->dev.inserted;
    if (inserted_box) *inserted_box = eng->dev.inserted_box;
    if (box7) *box7 = eng->box7.p;
    return r3d_check_launch("r3d_engine_inserted_device");
}

extern "C" int r3d_engine_set_world_aug(r3d_engine* eng, const r3d_world_aug* p) {
    if (!bind(eng)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_world_aug: null engine");
    if (!p) { eng->world_on = false; return R3D_OK; }
    const float v[5] = {p->flip_x_prob, p->flip_y_prob, p->rot_max, p->scale_lo, p->scale_hi};
    for (float x : v)
        if (!std::isfinite(x)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_world_aug: non-finite value");
    if (p->flip_x_prob < 0.f || p->flip_x_prob > 1.f || p->flip_y_prob < 0.f || p->flip_y_prob > 1.f)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_world_aug: flip probabilities must be in [0, 1]");
    if (p->rot_max < 0.f || p->rot_max > (float)kPi)                // pi as the float32 the caller passes
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_world_aug: rot_max must be in [0, pi]");
    if (!(p->scale_lo > 0.f) || p->scale_hi < p->scale_lo)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_world_aug: need 0 < scale_lo <= scale_hi");
    eng->world_pol = *p;
    eng->world_on = true;
    return R3D_OK;
}

extern "C" int r3d_engine_world_device(r3d_engine* eng, const float** params) {
    if (!bind(eng) || !params) return r3d_fail(R3D_ERR_ARG, "r3d_engine_world_device: null argument");
    if (!eng->batch_loaded || !eng->world_loaded)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_world_device: the batch was not loaded with a world augmentation");
    *params = eng->world.p;
    return R3D_OK;
}

extern "C" int r3d_engine_set_object_targets(r3d_engine* eng, const float* dims3, const int32_t* class_target) {
    if (!bind(eng) || !dims3 || !class_target || !eng->objects_set) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_object_targets: bad argument or no objects");
    const EngineDev& d = eng->dev;
    for (int c = 0; c < d.n_classes; ++c)
        if (class_target[c] < 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_set_object_targets: negative class id");
    TRY(eng->obj_dims3.alloc((size_t)d.n_objects * 3));
    TRY(eng->class_target.alloc((size_t)d.n_classes));
    R3D_CUDA(cudaMemcpy(eng->obj_dims3.p, dims3, (size_t)d.n_objects * 3 * sizeof(float), cudaMemcpyHostToDevice));
    R3D_CUDA(cudaMemcpy(eng->class_target.p, class_target, (size_t)d.n_classes * sizeof(int), cudaMemcpyHostToDevice));
    return R3D_OK;
}

extern "C" int r3d_engine_targets_device(r3d_engine* eng, const r3d_resident_store* s, const float* scene_box7,
                                         const int32_t* scene_class, int32_t max_targets, float* out_box7, int32_t* out_class,
                                         int32_t* out_count) {
    if (!bind(eng) || !s || !out_box7 || !out_class || !out_count) return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: null argument");
    if (!eng->ran) return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: run first");
    if (!eng->from_store) return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: the batch was not loaded from a resident store");
    const EngineDev& d = eng->dev;
    if (d.task != 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: detection targets need an object detection engine");
    if (!eng->obj_dims3.p) return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: set the object targets first");
    if (s->n_scans <= 0 || !s->box_offsets || !s->h_box_offsets)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: missing store arrays");
    const int total = s->h_box_offsets[s->n_scans];
    if (total > 0 && (!scene_box7 || !scene_class)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: missing scene targets");
    if (eng->kept_src != scene_class || (int)eng->kept.size() != s->n_scans) {
        std::vector<int> cls((size_t)total);
        if (total > 0) R3D_CUDA(cudaMemcpy(cls.data(), scene_class, (size_t)total * sizeof(int), cudaMemcpyDeviceToHost));
        eng->kept.assign(s->n_scans, 0);
        for (int i = 0; i < s->n_scans; ++i)
            for (int j = s->h_box_offsets[i]; j < s->h_box_offsets[i + 1]; ++j) eng->kept[i] += cls[j] != 0;
        eng->kept_src = scene_class;
    }
    int bound = 0;
    for (int i : eng->batch_idx) {
        if (i < 0 || i >= s->n_scans) return r3d_fail(R3D_ERR_ARG, "r3d_engine_targets_device: batch index outside this store");
        if ((long long)eng->kept[i] + d.max_events - 1 > max_targets)
            return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_targets_device: max_targets below a scan's kept scene boxes + max_events - 1");
        bound = std::max(bound, eng->kept[i] + d.max_events);
    }
    eng->targets_bound = bound;
    launch_gt_targets(eng->idx_dev.p, s->box_offsets, scene_box7, scene_class, eng->dev.st, eng->dev.inserted, eng->dev.inserted_box,
                      d.max_events, eng->obj_dims3.p, eng->class_target.p, eng->world_loaded ? eng->world.p : nullptr, eng->n_scans,
                      max_targets, out_box7, out_class, out_count, eng->stream);
    return r3d_check_launch("r3d_engine_targets_device");
}

extern "C" int r3d_engine_target_points_device(r3d_engine* eng, int32_t max_targets, float* box7, int32_t* cls, int32_t* count,
                                               int32_t min_points, int32_t* out_points, int32_t* out_point_gt) {
    if (!bind(eng) || !box7 || !cls || !count || !out_points || !out_point_gt)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_target_points_device: null argument");
    if (!eng->ran) return r3d_fail(R3D_ERR_ARG, "r3d_engine_target_points_device: run first");
    if (!eng->from_store)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_target_points_device: the batch was not loaded from a resident store");
    const EngineDev& d = eng->dev;
    if (d.task != 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_target_points_device: detection targets need an object detection engine");
    if (min_points < 0) return r3d_fail(R3D_ERR_ARG, "r3d_engine_target_points_device: min_points < 0");
    if (max_targets < 1) return r3d_fail(R3D_ERR_ARG, "r3d_engine_target_points_device: max_targets < 1");
    if (eng->targets_bound == 0)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_target_points_device: no r3d_engine_targets_device for this batch");
    const int cap = std::min(max_targets, eng->targets_bound);
    if (cap > TARGET_POINTS_MAX_BOXES)
        return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_target_points_device: more than 2048 targets in a scan");
    if (min_points > 0 && (size_t)d.B * (cap + 1) > eng->tp_remap.n) TRY(eng->tp_remap.alloc((size_t)d.B * (cap + 1)));
    R3D_CUDA(launch_target_points(eng->out_xyzi.p, eng->out_off.p, eng->n_scans, eng->max_n0 + d.max_inserted, box7, cls, count,
                                  max_targets, cap, min_points, out_points, out_point_gt, eng->tp_remap.p, eng->stream));
    return r3d_check_launch("r3d_engine_target_points_device");
}

extern "C" int r3d_engine_fetch(r3d_engine* eng, r3d_batch_result* res) {
    if (!bind(eng) || !res || !eng->ran) return r3d_fail(R3D_ERR_ARG, "r3d_engine_fetch: run first");
    EngineDev& d = eng->dev;
    const int n = eng->n_scans;
    cudaStream_t st = eng->stream;
    R3D_CUDA(engine_wait(eng));
    const long long total = eng->h_offsets[n], total_check = eng->h_offsets[d.B + 1 + n];
    if (total > res->capacity_points || total_check > res->capacity_check)
        return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_fetch: result buffers too small");
    if (res->out_offsets) memcpy(res->out_offsets, eng->h_offsets, (n + 1) * sizeof(long long));
    if (res->check_offsets) memcpy(res->check_offsets, eng->h_offsets + d.B + 1, (n + 1) * sizeof(long long));
    if (res->out_xyzi && total) R3D_CUDA(cudaMemcpyAsync(res->out_xyzi, eng->out_xyzi.p, (size_t)total * sizeof(float4), cudaMemcpyDeviceToHost, st));
    if (res->out_labels && total) R3D_CUDA(cudaMemcpyAsync(res->out_labels, eng->out_label.p, (size_t)total * sizeof(unsigned), cudaMemcpyDeviceToHost, st));
    if (res->out_labels16 && total) {                  // 16-bit labels over PCIe (widened again by the caller)
        if ((size_t)total > eng->out_label16.n) TRY(eng->out_label16.alloc((size_t)d.B * d.P));
        k_narrow_labels<<<eng->n_sms * 4, 256, 0, st>>>(eng->out_label.p, eng->out_label16.p, total); r3d_count_launch();
        R3D_CUDA(cudaMemcpyAsync(res->out_labels16, eng->out_label16.p, (size_t)total * sizeof(unsigned short), cudaMemcpyDeviceToHost, st));
    }
    if (res->check_xyzil && total_check) R3D_CUDA(cudaMemcpyAsync(res->check_xyzil, eng->out_check.p, (size_t)total_check * 5 * sizeof(float), cudaMemcpyDeviceToHost, st));
    if (res->inserted) R3D_CUDA(cudaMemcpyAsync(res->inserted, eng->dev.inserted, (size_t)n * d.max_events * 4 * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (res->inserted_box) R3D_CUDA(cudaMemcpyAsync(res->inserted_box, eng->dev.inserted_box, (size_t)n * d.max_events * 8 * sizeof(double), cudaMemcpyDeviceToHost, st));
    std::vector<ScanState> hs(n);
    R3D_CUDA(cudaMemcpyAsync(hs.data(), eng->dev.st, n * sizeof(ScanState), cudaMemcpyDeviceToHost, st));
    R3D_CUDA(engine_wait(eng));
    for (int s = 0; s < n; ++s) {
        if (res->n_inserted) res->n_inserted[s] = hs[s].n_inserted;
        if (res->status) res->status[s] = hs[s].status;
    }
    if (res->rounds) *res->rounds = eng->walked ? (int)eng->h_offsets[2 * (d.B + 1)] : eng->last_rounds;
    return R3D_OK;
}

extern "C" int r3d_engine_profile_enable(r3d_engine* eng, int on) {
    if (!bind(eng)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_profile_enable: null engine");
    cudaStreamSynchronize(eng->stream);
    drain_events(eng);
    eng->profile = on != 0;
    for (int i = 0; i < KID_COUNT; ++i) { eng->prof_ms[i] = 0; eng->prof_launches[i] = 0; }
    R3D_CUDA(cudaMemset(eng->stats.p, 0, R3D_N_STATS * sizeof(unsigned long long)));
    return R3D_OK;
}

extern "C" int r3d_engine_stats_ex(r3d_engine* eng, uint64_t* out, int n) {
    if (!bind(eng) || !out || n < 0 || n > R3D_N_STATS) return r3d_fail(R3D_ERR_ARG, "r3d_engine_stats_ex: bad argument");
    R3D_CUDA(cudaStreamSynchronize(eng->stream));
    R3D_CUDA(cudaMemcpy(out, eng->stats.p, (size_t)n * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return R3D_OK;
}

extern "C" int r3d_engine_walk_profile(r3d_engine* eng, int64_t* cycles, int32_t* tries, int n) {
    if (!bind(eng) || !cycles || !tries || n < 0 || n > eng->dev.B) return r3d_fail(R3D_ERR_ARG, "r3d_engine_walk_profile: bad argument");
    R3D_CUDA(cudaStreamSynchronize(eng->stream));
    std::vector<ScanState> st((size_t)n);
    R3D_CUDA(cudaMemcpy(st.data(), eng->dev.st, (size_t)n * sizeof(ScanState), cudaMemcpyDeviceToHost));
    for (int i = 0; i < n; ++i) { cycles[i] = st[i].walk_cycles; tries[i] = st[i].walk_tries; }
    return R3D_OK;
}

extern "C" int r3d_engine_stats(r3d_engine* eng, uint64_t* out8) {
    if (!bind(eng) || !out8) return r3d_fail(R3D_ERR_ARG, "r3d_engine_stats: null argument");
    R3D_CUDA(cudaStreamSynchronize(eng->stream));
    R3D_CUDA(cudaMemcpy(out8, eng->stats.p, 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    return R3D_OK;
}

extern "C" void* r3d_engine_stream(r3d_engine* eng) { return bind(eng) ? (void*)eng->stream : nullptr; }

extern "C" int r3d_engine_profile_read(r3d_engine* eng, char* names_out, int names_cap, double* ms_out,
                                       int64_t* launches_out, int max_kernels, int* n_kernels_out) {
    if (!bind(eng)) return r3d_fail(R3D_ERR_ARG, "r3d_engine_profile_read: null engine");
    cudaStreamSynchronize(eng->stream);
    drain_events(eng);
    std::string names;
    const int n = std::min<int>(KID_COUNT, max_kernels);
    for (int i = 0; i < n; ++i) {
        names += kKernelNames[i]; names += '\n';
        if (ms_out) ms_out[i] = eng->prof_ms[i];
        if (launches_out) launches_out[i] = eng->prof_launches[i];
    }
    if (names_out && names_cap > 0) { strncpy(names_out, names.c_str(), names_cap - 1); names_out[names_cap - 1] = 0; }
    if (n_kernels_out) *n_kernels_out = n;
    return R3D_OK;
}

extern "C" int r3d_engine_debug_image(r3d_engine* eng, int scan, double* smooth_out) {
    if (!bind(eng) || scan < 0 || scan >= eng->n_scans || !smooth_out) return r3d_fail(R3D_ERR_ARG, "r3d_engine_debug_image: bad argument");
    R3D_CUDA(cudaStreamSynchronize(eng->stream));
    R3D_CUDA(cudaMemcpy(smooth_out, eng->dev.smooth + (size_t)scan * eng->dev.hw, (size_t)eng->dev.hw * sizeof(double), cudaMemcpyDeviceToHost));
    return R3D_OK;
}

extern "C" int r3d_engine_debug_candidates(r3d_engine* eng, int scan, uint8_t* flags_out, double* level_out, int32_t* visible_out) {
    if (!bind(eng) || scan < 0 || scan >= eng->n_scans) return r3d_fail(R3D_ERR_ARG, "r3d_engine_debug_candidates: bad argument");
    const size_t K1 = eng->dev.K + 1;
    R3D_CUDA(cudaStreamSynchronize(eng->stream));
    if (flags_out) R3D_CUDA(cudaMemcpy(flags_out, eng->dev.cand_flags + scan * K1, K1, cudaMemcpyDeviceToHost));
    if (level_out) R3D_CUDA(cudaMemcpy(level_out, eng->dev.cand_level + scan * K1, K1 * sizeof(double), cudaMemcpyDeviceToHost));
    if (visible_out) R3D_CUDA(cudaMemcpy(visible_out, eng->dev.cand_v + scan * K1, K1 * sizeof(int), cudaMemcpyDeviceToHost));
    return R3D_OK;
}

extern "C" int r3d_engine_debug_col_index(r3d_engine* eng, int scan, int32_t* group_out, int32_t* off_out, int32_t* idx_out,
                                          uint16_t* col_out) {
    if (!bind(eng) || scan < 0 || scan >= eng->n_scans || !group_out) return r3d_fail(R3D_ERR_ARG, "r3d_engine_debug_col_index: bad argument");
    const EngineDev& d = eng->dev;
    const size_t ng1 = (size_t)col_groups(d.cols) + 1;
    *group_out = COL_GROUP;
    R3D_CUDA(cudaStreamSynchronize(eng->stream));
    if (off_out) R3D_CUDA(cudaMemcpy(off_out, d.col_off + scan * ng1, ng1 * sizeof(int), cudaMemcpyDeviceToHost));
    if (idx_out) R3D_CUDA(cudaMemcpy(idx_out, d.col_idx + (size_t)scan * d.max_points, (size_t)d.max_points * sizeof(int), cudaMemcpyDeviceToHost));
    if (col_out) R3D_CUDA(cudaMemcpy(col_out, d.col + (size_t)scan * d.P, (size_t)d.max_points * sizeof(uint16_t), cudaMemcpyDeviceToHost));
    return R3D_OK;
}

// ------------------------------------------------------------------------------- find_possible_places probe
namespace {

// the probed scan: originals stay resident for the road level but are not part of the "current scene"; the caller's
// rows become the (fp64) tail; one try is armed for `obj`
__global__ void k_probe_setup(EngineDev e, int n_scans, int scan, int obj, int n_rows) {
    const int b = blockIdx.x;
    if (b >= n_scans) return;
    ScanState& s = e.st[b];
    const bool me = b == scan;
    if (threadIdx.x == 0) {
        s.try_active = me; s.need_project = 0; s.apply_flag = 0; s.dirty = 0;
        e.gate_try[b] = me; e.gate_update[b] = me; e.gate_apply[b] = 0; e.gate_full[b] = 0; e.gate_patch[b] = 0;
        for (int i = 0; i < 4; ++i) e.tickets[(size_t)b * 4 + i] = 0u;
        if (me) {
            s.n_tail = n_rows; s.cur_obj = obj; s.cur_class = e.obj[obj].cls; s.n_feasible = 0; s.found_rank = INT_MAX;
            // the whole probed scene is one "inserted object" with an all-covering, zero-size box, so that k_collide
            // visits every tail point and no object point can ever be inside that box
            Box dummy;
            dummy.cx = dummy.cy = dummy.cz = 0.0;
            for (int i = 0; i < 9; ++i) dummy.m[i] = (i % 4 == 0) ? 1.0 : 0.0;
            dummy.length = dummy.width = dummy.height = 0.0; dummy.reach = 1e9;
            e.boxes[(size_t)b * e.max_boxes + s.n_boxes] = dummy;
            e.box_tests[(size_t)b * e.max_boxes + s.n_boxes] = make_box_test(dummy);
            e.inserted[((size_t)b * e.max_events + 0) * 4 + 3] = n_rows;
            s.n_boxes += 1; s.n_inserted = 1;
        }
    }
    if (!me) return;
    const int ww = e.map_window * e.map_window / 32;
    if (e.task == 1) for (int i = threadIdx.x; i < ww; i += blockDim.x) e.occ_win[(size_t)b * ww + i] = 0u;
    if (e.task == 1) occ_far_clear(e, b, threadIdx.x);
}

__global__ void k_probe_points(EngineDev e, int scan, int obj, int n_feasible, double* xyz_out, double* box_out) {
    const ObjBox ob = e.obj[obj];
    const size_t cb = (size_t)scan * (e.K + 1);
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k <= e.K; k += gridDim.x * blockDim.x) {
        const YawBox yb = make_yaw_box(ob.cx, ob.cy, ob.a, ob.b, e.cos_k[k], e.sin_k[k]);
        double* bo = box_out + (size_t)k * 5;
        bo[0] = yb.cx; bo[1] = yb.cy; bo[2] = e.cand_level[cb + k]; bo[3] = yb.m00; bo[4] = yb.m10;
    }
    if (!xyz_out) return;
    const long long total = (long long)n_feasible * ob.count;
    for (long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
        const int f = (int)(t / ob.count), i = (int)(t % ob.count);
        const int k = e.feas[(size_t)scan * e.K + f];
        const double c = e.cos_k[k], sn = e.sin_k[k];
        const double x0 = e.obj_x[ob.first + i], y0 = e.obj_y[ob.first + i];
        double* o = xyz_out + t * 3;
        o[0] = sub(mul(c, x0), mul(sn, y0));
        o[1] = add(mul(sn, x0), mul(c, y0));
        o[2] = add(e.obj_z[ob.first + i], sub(e.cand_level[cb + k], ob.cz));
    }
}

}  // namespace

extern "C" int r3d_engine_probe_places(r3d_engine* eng, int scan, int object_id, const double* scene_rows9, int64_t n_rows,
                                       uint8_t* flags_out, double* box_out, double* xyz_out, int xyz_capacity,
                                       int32_t* n_feasible_out) {
    if (!bind(eng) || !eng->batch_loaded || scan < 0 || scan >= eng->n_scans || object_id < 0 || object_id >= eng->dev.n_objects ||
        n_rows < 0 || (n_rows > 0 && !scene_rows9) || !flags_out || !box_out || !n_feasible_out)
        return r3d_fail(R3D_ERR_ARG, "r3d_engine_probe_places: bad argument");
    EngineDev d = eng->dev;
    if (n_rows > d.max_inserted) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_probe_places: scene larger than max_inserted");
    if (eng->h_nbox0[scan] + 1 > d.max_boxes) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_probe_places: max_boxes too small");
    const int n = eng->n_scans;
    cudaStream_t st = eng->stream;
    TRY(arm_batch(eng, false));
    // current scene -> fp64 tail of the probed scan; the original rows are not part of it
    std::vector<double> x(n_rows), y(n_rows), z(n_rows);
    std::vector<float> in(n_rows);
    std::vector<unsigned> lab(n_rows);
    for (int64_t i = 0; i < n_rows; ++i) {
        const double* p = scene_rows9 + i * 9;
        x[i] = p[0]; y[i] = p[1]; z[i] = p[2]; in[i] = (float)p[6]; lab[i] = (unsigned)(long long)p[7];
    }
    R3D_CUDA(cudaStreamSynchronize(st));
    std::vector<int> n0v(n);
    R3D_CUDA(cudaMemcpy(n0v.data(), eng->n0_arr.p, n * sizeof(int), cudaMemcpyDeviceToHost));
    const int n0 = n0v[scan];
    const size_t tb = (size_t)scan * d.max_inserted, pb = (size_t)scan * d.P;
    R3D_CUDA(cudaMemsetAsync(eng->dev.alive + pb, 0, n0, st));
    if (n_rows) {
        R3D_CUDA(cudaMemcpyAsync(eng->dev.tail_x + tb, x.data(), n_rows * sizeof(double), cudaMemcpyHostToDevice, st));
        R3D_CUDA(cudaMemcpyAsync(eng->dev.tail_y + tb, y.data(), n_rows * sizeof(double), cudaMemcpyHostToDevice, st));
        R3D_CUDA(cudaMemcpyAsync(eng->dev.tail_z + tb, z.data(), n_rows * sizeof(double), cudaMemcpyHostToDevice, st));
        R3D_CUDA(cudaMemcpyAsync(eng->dev.tail_i + tb, in.data(), n_rows * sizeof(float), cudaMemcpyHostToDevice, st));
        R3D_CUDA(cudaMemcpyAsync(eng->dev.label + pb + n0, lab.data(), n_rows * sizeof(unsigned), cudaMemcpyHostToDevice, st));
        R3D_CUDA(cudaMemsetAsync(eng->dev.alive + pb + n0, 1, n_rows, st));
    }
    k_probe_setup<<<n, 128, 0, st>>>(d, n, scan, object_id, (int)n_rows); r3d_count_launch();
    const int chunks_all = (n0 + (int)n_rows + CHUNK - 1) / CHUNK;
    if (d.task == 1) { k_adjust_map<<<dim3(chunks_all, n), STREAM_THREADS, 0, st>>>(d, n); r3d_count_launch(); }
    const int task_ctas = eng->n_sms * TASK_CTAS_PER_SM;
    const size_t pref_smem = (size_t)(n + 1) * sizeof(int);
    k_onmap<<<n, TRY_THREADS, onmap_smem_bytes(d.K), st>>>(d, n); r3d_count_launch();
    if (d.task == 0) { k_onmap_full<<<task_ctas, TASK_THREADS, pref_smem, st>>>(d, n, 0); r3d_count_launch(); }
    k_road_level<<<task_ctas, TASK_THREADS, pref_smem, st>>>(d, n, 0); r3d_count_launch();
    if (d.task == 1) { if (d.K <= SS_MAX_K) k_onmap_ss<<<n, 1024, 0, st>>>(d, n); else k_onmap_ss_seq<<<n, 1024, 0, st>>>(d, n); r3d_count_launch(); }
    k_collide<<<task_ctas, TASK_THREADS, pref_smem, st>>>(d, n, 0); r3d_count_launch();
    k_feasible_list<<<n, 128, 0, st>>>(d, n); r3d_count_launch();
    std::vector<ScanState> hs(1);
    R3D_CUDA(cudaMemcpyAsync(hs.data(), eng->dev.st + scan, sizeof(ScanState), cudaMemcpyDeviceToHost, st));
    R3D_CUDA(cudaStreamSynchronize(st));
    const int nf = hs[0].n_feasible;
    *n_feasible_out = nf;
    if (hs[0].status != 0) return r3d_fail(hs[0].status, "r3d_engine_probe_places: scan status");
    if (xyz_out && nf > xyz_capacity) return r3d_fail(R3D_ERR_CAPACITY, "r3d_engine_probe_places: xyz_capacity too small");
    const size_t K1 = d.K + 1;
    DevBuf<double> dbox, dxyz;
    TRY(dbox.alloc(K1 * 5));
    std::vector<ObjBox> hob(1);
    R3D_CUDA(cudaMemcpy(hob.data(), eng->obj.p + object_id, sizeof(ObjBox), cudaMemcpyDeviceToHost));
    const size_t nxyz = xyz_out ? (size_t)nf * hob[0].count * 3 : 0;
    if (nxyz) TRY(dxyz.alloc(nxyz));
    k_probe_points<<<148, 256, 0, st>>>(d, scan, object_id, nf, nxyz ? dxyz.p : nullptr, dbox.p); r3d_count_launch();
    R3D_CUDA(cudaMemcpyAsync(flags_out, eng->dev.cand_flags + scan * K1, K1, cudaMemcpyDeviceToHost, st));
    R3D_CUDA(cudaMemcpyAsync(box_out, dbox.p, K1 * 5 * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (nxyz) R3D_CUDA(cudaMemcpyAsync(xyz_out, dxyz.p, nxyz * sizeof(double), cudaMemcpyDeviceToHost, st));
    R3D_CUDA(cudaStreamSynchronize(st));
    return r3d_check_launch("r3d_engine_probe_places");
}
