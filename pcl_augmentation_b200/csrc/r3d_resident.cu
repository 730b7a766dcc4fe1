// Kernels of the resident-dataset path (r3d_engine_load_resident, include/real3d_b200.h): batches gathered from a
// dataset that already sits in device memory, and their schedules drawn on the device, so that augmenting a new batch
// moves no per-point byte over PCIe and needs no host round trip for its randomness.
#include "r3d_resident.h"
#include "r3d_host.h"

namespace r3d {

constexpr int GATHER_CHUNK = 4096;       // points per CTA: the (chunk, scan) grid of k_widen_labels
constexpr int GATHER_THREADS = 256;
constexpr int DRAW_WARPS = 4;            // warps per CTA of k_draw_schedule

// ------------------------------------------------------------------------------------------------ gathers
// A pure copy: per point one 16-byte load + store of xyzi and a 2-byte label read widened to the engine's u32 row.
__global__ void __launch_bounds__(GATHER_THREADS) k_gather_points(const float4* __restrict__ src_xyzi,
                                                                  const unsigned short* __restrict__ src_label,
                                                                  const long long* __restrict__ pt_off, const int* __restrict__ idx,
                                                                  float4* __restrict__ xyzi, int max_points,
                                                                  unsigned* __restrict__ label, int P, int od, unsigned road_label) {
    const int b = blockIdx.y;
    const int s = __ldg(idx + b);
    const long long o = __ldg(pt_off + s);
    const int cnt = (int)(__ldg(pt_off + s + 1) - o);
    const int p0 = blockIdx.x * GATHER_CHUNK;
    const int p1 = min(p0 + GATHER_CHUNK, cnt);
    const unsigned other = road_label == 1u ? 2u : 1u;       // od/ins:353-355 relabels every non-Road point to 1
    float4* dx = xyzi + (size_t)b * max_points;
    unsigned* dl = label + (size_t)b * P;
    for (int p = p0 + threadIdx.x; p < p1; p += GATHER_THREADS) {
        __stcs(dx + p, __ldcs(src_xyzi + o + p));            // streamed once: keep them out of the way of L2 residents
        unsigned l = __ldcs(src_label + o + p);
        if (od) l = l == road_label ? road_label : other;
        dl[p] = l;
    }
}

// one thread per scan: point / box counts, OD map offsets + dims (the maps stay in the store) or the semseg pose
__global__ void k_gather_scan_meta(r3d_resident_store s, const int* __restrict__ idx, int n, int od, int* n0, int* nbox0,
                                   long long* map_off, int* map_dims, double* poses) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const int i = idx[b];
    n0[b] = (int)(s.point_offsets[i + 1] - s.point_offsets[i]);
    nbox0[b] = s.box_offsets[i + 1] - s.box_offsets[i];
    if (od) {
        map_off[2 * b] = s.map_offsets[2 * i];
        map_off[2 * b + 1] = s.map_offsets[2 * i + 1];
        for (int k = 0; k < 8; ++k) map_dims[8 * b + k] = s.map_dims[8 * i + k];
    } else {
        for (int k = 0; k < 16; ++k) poses[16 * b + k] = s.poses[16 * i + k];
    }
}

// the scene boxes of scan b into its max_boxes slots (zeros past the scan's boxes, as r3d_engine_load_batch leaves
// them); a Box is the 16-double record, moved as 8 x 16 bytes
__global__ void k_gather_boxes(const double2* __restrict__ src, const int* __restrict__ box_off, const int* __restrict__ idx,
                               double2* boxes, double2* boxes0, int max_boxes) {
    const int b = blockIdx.y;
    const int i = idx[b];
    const int first = box_off[i], nb = box_off[i + 1] - first;
    const int words = max_boxes * 8;
    for (int t = blockIdx.x * blockDim.x + threadIdx.x; t < words; t += gridDim.x * blockDim.x) {
        const int j = t >> 3;
        const double2 v = j < nb ? src[(size_t)first * 8 + t] : make_double2(0.0, 0.0);
        boxes[(size_t)b * words + t] = v;
        boxes0[(size_t)b * words + t] = v;
    }
}

// ------------------------------------------------------------------------------------------- schedule draw
// Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011): a keyed bijection of a
// 128-bit counter, so any (key, counter) gives its draws directly and no generator state is carried anywhere.
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const unsigned hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const unsigned hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += 0x9E3779B9u; k.y += 0xBB67AE85u;
    }
    return c;
}
// unbiased integer in [0, range) from one 32-bit word (Lemire, "Fast random integer generation in an interval", 2019):
// false when the word falls in the biased part and has to be rejected
__device__ __forceinline__ bool bounded(unsigned x, unsigned range, unsigned& v) {
    const unsigned long long m = (unsigned long long)x * range;
    v = (unsigned)(m >> 32);
    const unsigned low = (unsigned)m;
    return low >= range || low >= (0u - range) % range;
}
__device__ __forceinline__ unsigned word_of(const uint4& w, int k) { return k == 0 ? w.x : k == 1 ? w.y : k == 2 ? w.z : w.w; }

// One warp per (scan, event, class) writes the head of that shuffle: the first k = min(T, n_c) entries of a uniform
// shuffle of [0, n_c) (a uniformly random ordered k-subset), then -1.  A partial Fisher-Yates shuffle: step j swaps
// position j with a uniform position r_j in [j, n_c).  Only the positions some step moved are kept, as a (position,
// value) list of at most k entries in shared memory searched by the whole warp, so the cost is k steps whatever n_c is
// (rejecting repeats of a uniform draw instead needs ~n_c ln n_c draws when k = n_c).  One more warp per scan draws the
// class counts.
// Streams: key = (seed low word, seed high word ^ epoch high word), counter = (c0, stream id, store index, epoch low
// word) with stream id 0 = counts (c0 = draw round * 32 + lane) and 1 + event * 16 + class = a head (c0 = step j, plus
// attempt << 16 for the rare words Lemire's method rejects).
__global__ void __launch_bounds__(DRAW_WARPS * 32) k_draw_schedule(const int* __restrict__ idx, int n, int E, int C, int T,
                                                                   const int* __restrict__ class_list_off, SchedulePolicy pol,
                                                                   unsigned long long seed, unsigned long long epoch,
                                                                   int* counts, int* perms) {
    extern __shared__ int s_head_all[];
    const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
    const long long w = (long long)blockIdx.x * DRAW_WARPS + wib;
    const int per_scan = E * C + 1;
    if (w >= (long long)n * per_scan) return;                // whole warps only: no warp-level call below sees a partial warp
    const int b = (int)(w / per_scan), r = (int)(w % per_scan);
    const unsigned sidx = (unsigned)idx[b];
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32) ^ (unsigned)(epoch >> 32));
    if (r == E * C) {                                        // class counts (generate_seed)
        int mine = 0;                                        // lane c accumulates class c
        if (pol.random) {
            int taken = 0;
            for (unsigned round = 0; taken < pol.number_of_object; ++round) {
                const uint4 x = philox4x32_10(make_uint4(round * 32u + lane, 0u, sidx, (unsigned)epoch), key);
                for (int k = 0; k < 4 && taken < pol.number_of_object; ++k) {
                    unsigned v;
                    const bool ok = bounded(word_of(x, k), (unsigned)C, v);
                    const unsigned okm = __ballot_sync(0xffffffffu, ok);
                    const int before = __popc(okm & ((1u << lane) - 1u));
                    const bool take = ok && taken + before < pol.number_of_object;
                    for (int c = 0; c < C; ++c) {
                        const int got = __popc(__ballot_sync(0xffffffffu, take && (int)v == c));
                        if (lane == c) mine += got;
                    }
                    taken += min(__popc(okm), pol.number_of_object - taken);
                }
            }
        } else {
#pragma unroll
            for (int c = 0; c < R3D_MAX_CLASSES; ++c) if (c == lane) mine = pol.fixed[c];   // constant indices: no local copy
        }
        if (lane < C) counts[(size_t)b * C + lane] = mine;
        return;
    }
    const int ev = r / C, c = r % C;
    const int nc = class_list_off[c + 1] - class_list_off[c];
    const int k = min(T, nc);
    int* rs = s_head_all + wib * 3 * T;           // r_j, then the head itself
    int* mkey = rs + T;                           // moved positions ...
    int* mval = mkey + T;                         // ... and the value each holds now
    const unsigned stream = 1u + (unsigned)ev * R3D_MAX_CLASSES + (unsigned)c;
    for (int j = lane; j < k; j += 32) {          // r_j = j + uniform [0, n_c - j)
        unsigned v = 0;
        bool ok = false;
        for (unsigned att = 0; !ok; ++att) {
            const uint4 x = philox4x32_10(make_uint4((unsigned)j | (att << 16), stream, sidx, (unsigned)epoch), key);
            for (int q = 0; q < 4 && !ok; ++q) ok = bounded(word_of(x, q), (unsigned)(nc - j), v);
        }
        rs[j] = j + (int)v;
    }
    __syncwarp();
    int nmap = 0;
    for (int j = 0; j < k; ++j) {
        const int rj = rs[j];
        int va = j, vb = rj, slot = -1;
        bool fa = false, fb = false;
        for (int t = lane; t < nmap; t += 32) {
            const int key_t = mkey[t];
            if (key_t == j) { va = mval[t]; fa = true; }
            if (key_t == rj) { vb = mval[t]; fb = true; slot = t; }
        }
        const unsigned ba = __ballot_sync(0xffffffffu, fa), bb = __ballot_sync(0xffffffffu, fb);
        if (ba) va = __shfl_sync(0xffffffffu, va, __ffs(ba) - 1);
        if (bb) { vb = __shfl_sync(0xffffffffu, vb, __ffs(bb) - 1); slot = __shfl_sync(0xffffffffu, slot, __ffs(bb) - 1); }
        if (lane == 0) {
            rs[j] = vb;                           // position j is final: the j-th entry of the shuffle
            if (rj != j) {                        // position rj now holds what position j held
                if (slot >= 0) mval[slot] = va;
                else { mkey[nmap] = rj; mval[nmap] = va; }
            }
        }
        if (rj != j && slot < 0) ++nmap;
        __syncwarp();
    }
    int* out = perms + (((size_t)b * E + ev) * C + c) * T;
    for (int j = lane; j < T; j += 32) out[j] = j < k ? rs[j] : -1;
}

// ------------------------------------------------------------------------------------------ detection targets
// per inserted object the float32 box (x, y, z_bottom, length, width, height, yaw) from inserted_box
// (cx cy cz m00 m10 length width height); rows past the scan's n_inserted are zero
__global__ void k_inserted_targets(const ScanState* __restrict__ sts, const double* __restrict__ ibox, int n, int E,
                                   int* n_inserted, float* box7) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n * E) return;
    const int b = t / E, j = t % E;
    const int ni = sts[b].n_inserted;
    if (j == 0) n_inserted[b] = ni;
    const double* q = ibox + (size_t)t * 8;
    float* o = box7 + (size_t)t * 7;
    const bool live = j < ni;
    o[0] = live ? (float)q[0] : 0.f; o[1] = live ? (float)q[1] : 0.f; o[2] = live ? (float)q[2] : 0.f;
    o[3] = live ? (float)q[5] : 0.f; o[4] = live ? (float)q[6] : 0.f; o[5] = live ? (float)q[7] : 0.f;
    o[6] = live ? (float)atan2(q[4], q[3]) : 0.f;
}

// ------------------------------------------------------------------------------------------ world augmentation
// One thread per scan: one Philox call on the stream id 0xFFFFFFFF (the schedule streams are 0 and 1 + event * 16 +
// class < 2^16), so the world parameters of a scan depend on (seed, epoch, store index) only.
__device__ __forceinline__ float uniform24(unsigned w) { return (float)(w >> 8) * 0x1p-24f; }   // exact, in [0, 1)

__global__ void k_draw_world(const int* __restrict__ idx, int n, r3d_world_aug pol, unsigned long long seed,
                             unsigned long long epoch, float* world) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= n) return;
    const uint2 key = make_uint2((unsigned)seed, (unsigned)(seed >> 32) ^ (unsigned)(epoch >> 32));
    const uint4 x = philox4x32_10(make_uint4(0u, 0xFFFFFFFFu, (unsigned)idx[b], (unsigned)epoch), key);
    const float theta = __fmul_rn(pol.rot_max, __fsub_rn(__fmul_rn(2.f, uniform24(x.z)), 1.f));
    const float k = __fadd_rn(pol.scale_lo, __fmul_rn(__fsub_rn(pol.scale_hi, pol.scale_lo), uniform24(x.w)));
    float* w = world + (size_t)b * 8;
    w[0] = uniform24(x.x) < pol.flip_x_prob ? 1.f : 0.f;
    w[1] = uniform24(x.y) < pol.flip_y_prob ? 1.f : 0.f;
    w[2] = theta; w[3] = cosf(theta); w[4] = sinf(theta); w[5] = k; w[6] = 0.f; w[7] = 0.f;
}

// ------------------------------------------------------------------------------------------ detection targets
__device__ __forceinline__ double wrap_pi(double h) {        // into [-pi, pi)
    return __dsub_rn(h, __dmul_rn(2.0 * kPi, floor(__dmul_rn(__dadd_rn(h, kPi), 1.0 / (2.0 * kPi)))));
}
// a target box through the scan's world transform (centre as the points, dimensions * k, heading flipped / rotated)
__device__ __forceinline__ void world_box(const WorldXf& t, float theta, float* o) {
    world_point(t, o[0], o[1], o[2]);
    o[3] = __fmul_rn(o[3], t.k); o[4] = __fmul_rn(o[4], t.k); o[5] = __fmul_rn(o[5], t.k);
    double h = (double)o[6];
    if (t.fx) h = -h;
    if (t.fy) h = -__dadd_rn(h, kPi);
    o[6] = (float)wrap_pi(__dadd_rn(h, (double)theta));
}

// One warp per scan writes its targets row: the kept scene boxes of its store scan, then its kept inserted objects,
// compacted with ballots, then zeros up to max_targets.  Inserted box: centre from inserted_box (cx cy cz_bottom m00
// m10 ...), z to the box centre with the cut object's unpadded height, heading atan2(m10, m00) - pi/2.
__global__ void k_gt_targets(const int* __restrict__ idx, const int* __restrict__ box_off, const float* __restrict__ scene_box7,
                             const int* __restrict__ scene_class, const ScanState* __restrict__ sts, const int* __restrict__ inserted,
                             const double* __restrict__ ibox, int E, const float* __restrict__ dims3,
                             const int* __restrict__ class_target, const float* __restrict__ world, int n, int max_targets,
                             float* out_box7, int* out_class, int* out_count) {
    const int b = (int)((blockIdx.x * (size_t)blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (b >= n) return;                                       // whole warps: n * 32 threads of whole CTAs
    const int i = idx[b];
    const int first = box_off[i], nb = box_off[i + 1] - first;
    const int ni = sts[b].n_inserted;
    float* ob = out_box7 + (size_t)b * max_targets * 7;
    int* oc = out_class + (size_t)b * max_targets;
    WorldXf wx{};
    float theta = 0.f;
    if (world) { wx = world_xf(world + (size_t)b * 8); theta = world[(size_t)b * 8 + 2]; }
    const unsigned below = (1u << lane) - 1u;
    int m = 0;
    for (int j0 = 0; j0 < nb; j0 += 32) {
        const int j = j0 + lane;
        const int cls = j < nb ? scene_class[first + j] : 0;
        const unsigned keep = __ballot_sync(0xffffffffu, cls != 0);
        if (cls != 0) {
            const int pos = m + __popc(keep & below);
            float o[7];
            for (int q = 0; q < 7; ++q) o[q] = scene_box7[(size_t)(first + j) * 7 + q];
            if (world) world_box(wx, theta, o);
            for (int q = 0; q < 7; ++q) ob[(size_t)pos * 7 + q] = o[q];
            oc[pos] = cls;
        }
        m += __popc(keep);
    }
    for (int j0 = 0; j0 < ni; j0 += 32) {
        const int j = j0 + lane;
        const size_t t = (size_t)b * E + j;
        const int cls = j < ni ? class_target[inserted[t * 4 + 2]] : 0;
        const unsigned keep = __ballot_sync(0xffffffffu, cls != 0);
        if (cls != 0) {
            const int pos = m + __popc(keep & below);
            const double* q = ibox + t * 8;
            const float* dm = dims3 + (size_t)inserted[t * 4] * 3;
            float o[7];
            o[0] = (float)q[0]; o[1] = (float)q[1];
            o[2] = (float)__dadd_rn(q[2], __dmul_rn((double)dm[2], 0.5));
            o[3] = dm[0]; o[4] = dm[1]; o[5] = dm[2];
            o[6] = (float)wrap_pi(__dsub_rn(atan2(q[4], q[3]), 0.5 * kPi));
            if (world) world_box(wx, theta, o);
            for (int r = 0; r < 7; ++r) ob[(size_t)pos * 7 + r] = o[r];
            oc[pos] = cls;
        }
        m += __popc(keep);
    }
    for (int p = m + lane; p < max_targets; p += 32) {
        for (int q = 0; q < 7; ++q) ob[(size_t)p * 7 + q] = 0.f;
        oc[p] = 0;
    }
    if (lane == 0) out_count[b] = m;
}

// ------------------------------------------------------------------------------------------------ launchers
void launch_gather_points(const r3d_resident_store& s, const int* idx, int n, int max_n0, float4* xyzi, int max_points,
                          unsigned* label, int P, int od, unsigned road_label, cudaStream_t st) {
    const int chunks = (max_n0 + GATHER_CHUNK - 1) / GATHER_CHUNK;
    k_gather_points<<<dim3(chunks, n), GATHER_THREADS, 0, st>>>(reinterpret_cast<const float4*>(s.xyzi), s.labels,
                                                                 reinterpret_cast<const long long*>(s.point_offsets), idx, xyzi,
                                                                 max_points, label, P, od, road_label);
    r3d_count_launch();
}

void launch_gather_meta(const r3d_resident_store& s, const int* idx, int n, int od, int* n0, int* nbox0, long long* map_off,
                        int* map_dims, double* poses, Box* boxes, Box* boxes0, int max_boxes, cudaStream_t st) {
    k_gather_scan_meta<<<(n + 127) / 128, 128, 0, st>>>(s, idx, n, od, n0, nbox0, map_off, map_dims, poses);
    const int words = max_boxes * 8;
    k_gather_boxes<<<dim3((words + 255) / 256, n), 256, 0, st>>>(reinterpret_cast<const double2*>(s.boxes), s.box_offsets, idx,
                                                                 reinterpret_cast<double2*>(boxes), reinterpret_cast<double2*>(boxes0),
                                                                 max_boxes);
    r3d_count_launch(2);
}

size_t draw_schedule_smem(int T) { return (size_t)DRAW_WARPS * 3 * T * sizeof(int); }
static_assert(DRAW_WARPS * 3 * DRAW_MAX_TRIES * sizeof(int) <= 200 * 1024 && DRAW_MAX_TRIES < (1 << 16),
              "DRAW_MAX_TRIES: the schedule draw's shared memory and its step counter word");

cudaError_t allow_draw_schedule_smem(int T) {
    cudaFuncAttributes a;
    cudaError_t err = cudaFuncGetAttributes(&a, k_draw_schedule);
    if (err != cudaSuccess || (size_t)a.maxDynamicSharedSizeBytes >= draw_schedule_smem(T)) return err;
    return cudaFuncSetAttribute(k_draw_schedule, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)draw_schedule_smem(T));
}

void launch_draw_schedule(const int* idx, int n, int E, int C, int T, const int* class_list_off, const SchedulePolicy& pol,
                          unsigned long long seed, unsigned long long epoch, int* counts, int* perms, cudaStream_t st) {
    const long long warps = (long long)n * (E * C + 1);
    const int blocks = (int)((warps + DRAW_WARPS - 1) / DRAW_WARPS);
    k_draw_schedule<<<blocks, DRAW_WARPS * 32, draw_schedule_smem(T), st>>>(idx, n, E, C, T, class_list_off, pol, seed, epoch,
                                                                            counts, perms);
    r3d_count_launch();
}

void launch_inserted_targets(const ScanState* sts, const double* inserted_box, int n, int E, int* n_inserted, float* box7,
                             cudaStream_t st) {
    k_inserted_targets<<<(n * E + 127) / 128, 128, 0, st>>>(sts, inserted_box, n, E, n_inserted, box7);
    r3d_count_launch();
}

void launch_draw_world(const int* idx, int n, const r3d_world_aug& pol, unsigned long long seed, unsigned long long epoch,
                       float* world, cudaStream_t st) {
    k_draw_world<<<(n + 127) / 128, 128, 0, st>>>(idx, n, pol, seed, epoch, world);
    r3d_count_launch();
}

void launch_gt_targets(const int* idx, const int* box_off, const float* scene_box7, const int* scene_class, const ScanState* sts,
                       const int* inserted, const double* inserted_box, int E, const float* dims3, const int* class_target,
                       const float* world, int n, int max_targets, float* out_box7, int* out_class, int* out_count,
                       cudaStream_t st) {
    constexpr int WARPS = 4;
    k_gt_targets<<<(n + WARPS - 1) / WARPS, WARPS * 32, 0, st>>>(idx, box_off, scene_box7, scene_class, sts, inserted, inserted_box,
                                                                  E, dims3, class_target, world, n, max_targets, out_box7,
                                                                  out_class, out_count);
    r3d_count_launch();
}

}  // namespace r3d
