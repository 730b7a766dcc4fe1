// Kernels of the batched Real3D-Aug engine, part: A11 / A12 slot update, A2 / A3 full re-projection, semseg map adjustment.
// Included by r3d_engine_kernels.cuh (inside namespace r3d, after the shared constants); not a standalone header.
// ------------------------------------------------------------------------------- apply mask + min/max el
__device__ __forceinline__ bool pix_removed(const EngineDev& e, int b, const ScanState& s, int pix) {
    if (pix < 0) return false;
    if (e.dmask[(size_t)b * e.dwords + (pix >> 5)] & (1u << (pix & 31))) return true;
    // od/ins:486: an empty object pixel holds 500, so scene pixels farther than 500 count as covered
    return e.far_arr[b] && e.smooth[(size_t)b * e.hw + pix] > kEmptyRange;
}

// Slot update, one CTA per scan (A11/A12 + the decision how the range image is refreshed):
//  1. scene = scene[pix_id not in vis_px] (od/ins:488-501, 545).  vis_px lies inside the pixel rectangle select_emit
//     recorded, so only the points whose azimuth bin falls in the column groups of that range are visited (CSR by
//     COL_GROUP columns, built once per scan) plus the inserted tail: O(window) instead of O(N).  Notes whether a
//     removed point held the scene's min / max elevation.
//  2. full re-projection or in-place patch?  The image geometry (od/ins:97-98) depends only on the scene's min / max
//     elevation; if neither moved, every surviving point keeps its pixel and only the pixels of vis_px change.
//  3. patch: the z-buffer changes only at the pixels of vis_px — all their scene points were removed (od/ins:491)
//     and the visible object points were appended there (od/ins:545).
constexpr int UPDATE_THREADS = 256;
#ifndef R3D_UPDATE_G
#define R3D_UPDATE_G 8
#endif
constexpr int UPDATE_G = R3D_UPDATE_G;   // CTAs per scan; the last one to finish takes the decision and patches
__device__ __forceinline__ bool last_block_done(unsigned* ticket, unsigned n_blocks) {
    __shared__ bool s_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(ticket, 1u) == n_blocks - 1;
    __syncthreads();
    if (s_last) __threadfence();
    return s_last;
}

// scene = scene[pix_id not in vis_px] (od/ins:488-501) for the calling thread's share (tid of nthr) of the points in
// the column range of the recorded rectangle + the inserted tail; true if a removed point held the min / max elevation
__device__ __forceinline__ void adjust_map_point(const EngineDev& e, int b, ScanState& s, const double* T, int p, int delta = 0,
                                                 bool ignore_alive = false);

template <bool OCC_COUNTS = false>      // OCC_COUNTS (walker, semseg): a removed point also leaves its map cell's count
__device__ __forceinline__ bool apply_vis_mask(const EngineDev& e, int b, ScanState& s, int tid, int nthr) {
    const double* T = e.poses + (size_t)b * 16;
    const size_t base = (size_t)b * e.P;
    bool extreme = false;
    const int* off = e.col_off + (size_t)b * (col_groups(e.cols) + 1);
    const int* idx = e.col_idx + (size_t)b * e.max_points;
    int c0 = s.d_c0, c1 = s.d_c1;
    if (e.far_arr[b]) { c0 = 0; c1 = e.cols - 1; }          // od/ins:486 quirk: covered pixels can be anywhere
    const unsigned long long lo = s.min_el_bits, hi = s.max_el_bits;
    if (c1 >= c0) {
        const int g0 = c0 / COL_GROUP, g1 = c1 / COL_GROUP;                 // the column groups that hold c0 .. c1
        const int beg = g0 > 0 ? off[g0 - 1] : 0, end = off[g1];           // off[g] = END of group g's bucket
        // index -> alive / pix -> mask word is a chain of dependent loads: four points per thread in flight
        for (int i = beg + tid; i < end; i += 4 * nthr) {
            int p[4], px[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) p[u] = i + u * nthr < end ? idx[i + u * nthr] : -1;
#pragma unroll
            for (int u = 0; u < 4; ++u) px[u] = (p[u] >= 0 && e.alive[base + p[u]]) ? e.pix[base + p[u]] : -1;
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (px[u] >= 0 && pix_removed(e, b, s, px[u])) {
                    e.alive[base + p[u]] = 0;
                    if (OCC_COUNTS) adjust_map_point(e, b, s, T, p[u], -1, true);
                    const unsigned long long bits = dbl_bits(e.el[base + p[u]]);
                    extreme |= bits == lo || bits == hi;
                }
        }
    }
    for (int t = tid; t < s.tail_before; t += nthr) {
        const int p = s.n0 + t;
        if (e.alive[base + p] && pix_removed(e, b, s, e.pix[base + p])) {
            e.alive[base + p] = 0;
            if (OCC_COUNTS) adjust_map_point(e, b, s, T, p, -1, true);
            const unsigned long long bits = dbl_bits(e.el[base + p]);
            extreme |= bits == lo || bits == hi;
        }
    }
    return extreme;
}

__global__ void __launch_bounds__(UPDATE_THREADS) k_update(EngineDev e, int n_scans) {
    const int b = blockIdx.y;
    if (b >= n_scans) return;
    const int do_apply = e.gate_apply[b], do_update = e.gate_update[b];
    if (!do_apply && !do_update) {
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            e.gate_full[b] = 0; e.gate_patch[b] = 0;
            int* r = e.cf_rect + (size_t)b * 4; r[0] = 0; r[1] = -1; r[2] = 0; r[3] = -1;
        }
        return;
    }
    ScanState& s = e.st[b];
    const size_t base = (size_t)b * e.P;
    const int tid = blockIdx.x * UPDATE_THREADS + threadIdx.x, nthr = UPDATE_G * UPDATE_THREADS;
    const bool extreme = do_apply && apply_vis_mask(e, b, s, tid, nthr);
    if (__syncthreads_or(extreme) && threadIdx.x == 0) atomicOr(&s.extreme_removed, 1);
    if (!last_block_done(&e.tickets[(size_t)b * 4 + 0], UPDATE_G)) return;
    __shared__ int s_patch;
    if (threadIdx.x == 0) {
        int full = 0, patch = 0;
        int* rect = e.cf_rect + (size_t)b * 4;
        rect[0] = 0; rect[1] = -1; rect[2] = 0; rect[3] = -1;
        if (do_update) {
            const bool extended = s.new_min_bits < s.min_el_bits || s.new_max_bits > s.max_el_bits;
            full = s.first || *(volatile int*)&s.extreme_removed || extended || e.far_arr[b] || e.force_full;
            patch = !full;
            if (full) {
                s.min_el_bits = R3D_EMPTY_U64; s.max_el_bits = 0ull;
                rect[0] = 0; rect[1] = e.rows - 1; rect[2] = 0; rect[3] = e.cols - 1;
            } else {
                rect[0] = max(s.d_r0 - 4, 0); rect[1] = min(s.d_r1 + 4, e.rows - 1);
                rect[2] = max(s.d_c0 - 2, 0); rect[3] = min(s.d_c1 + 2, e.cols - 1);
            }
            s.first = 0;
            s.new_min_bits = R3D_EMPTY_U64; s.new_max_bits = 0ull;
            atomicAdd(&e.stats[full ? 0 : 3], 1ull);
        }
        s.extreme_removed = 0;
        e.gate_full[b] = full; e.gate_patch[b] = patch;
        s_patch = patch;
        if (full) e.full_list[atomicAdd(&e.work_cnt[0], 1)] = b;
        if (rect[1] >= rect[0] && rect[3] >= rect[2]) {             // close/fill tiles that overlap the rectangle
            const int ty0 = rect[0] / CF_TH, ty1 = rect[1] / CF_TH, tx0 = rect[2] / CF_TW, tx1 = rect[3] / CF_TW;
            const int nt = (ty1 - ty0 + 1) * (tx1 - tx0 + 1);
            int* task = e.cf_tasks + atomicAdd(&e.work_cnt[1], nt);
            for (int ty = ty0; ty <= ty1; ++ty)
                for (int tx = tx0; tx <= tx1; ++tx) *task++ = b * e.cf_tiles + ty * e.cf_tiles_x + tx;
        }
    }
    __syncthreads();
    if (do_update && e.task == 1) {
        const int ww = e.map_window * e.map_window / 32;
        unsigned* o = e.occ_win + (size_t)b * ww;
        for (int i = threadIdx.x; i < ww; i += UPDATE_THREADS) o[i] = 0u;
        occ_far_clear(e, b, threadIdx.x);
    }
    if (!s_patch) return;
    unsigned long long* z = e.zraw + (size_t)b * e.hw;
    const unsigned* dm = e.dmask + (size_t)b * e.dwords;
    if (s.d_r1 >= s.d_r0 && s.d_c1 >= s.d_c0) {
        // vis_px lies inside the rectangle select_emit recorded: visit only the mask words that hold its columns, row
        // by row (a word may be visited for two rows when the width is no multiple of 32; clearing twice is harmless)
        const int nw = (s.d_c1 >> 5) - (s.d_c0 >> 5) + 2, nrow = s.d_r1 - s.d_r0 + 1;
        for (int i = threadIdx.x; i < nrow * nw; i += UPDATE_THREADS) {
            const int r = s.d_r0 + i / nw;
            const int w = ((r * e.cols + s.d_c0) >> 5) + i % nw;
            if (w > ((r * e.cols + s.d_c1) >> 5)) continue;
            unsigned m = dm[w];
            while (m) { const int bit = __ffs(m) - 1; m &= m - 1; z[(w << 5) + bit] = R3D_EMPTY_U64; }
        }
    }
    __syncthreads();
    if (s.apply_flag)                                        // points appended by the accept being applied
        for (int p = s.n0 + s.tail_before + threadIdx.x; p < s.n0 + s.n_tail; p += UPDATE_THREADS)
            if (e.alive[base + p]) atomicMin(&z[e.pix[base + p]], dbl_bits(e.r[base + p]));
}

// A2 (od/ins:79-80) on the cached elevations: min / max over the live points (full path only)
__global__ void __launch_bounds__(STREAM_THREADS) k_minmax(EngineDev e, int n_scans) {
    __shared__ unsigned long long s_min[STREAM_THREADS / 32], s_max[STREAM_THREADS / 32];
    const int n_full = e.work_cnt[0];
    for (int li = blockIdx.y; li < n_full; li += gridDim.y) {       // the scans k_update listed for a full re-projection
    const int b = e.full_list[li];
    ScanState& s = e.st[b];
    const int n = s.n0 + s.n_tail;
    const int p0 = blockIdx.x * CHUNK;
    if (p0 >= n) continue;
    const size_t base = (size_t)b * e.P;
    unsigned long long lmin = R3D_EMPTY_U64, lmax = 0ull;
    for (int p = p0 + threadIdx.x; p < min(p0 + CHUNK, n); p += STREAM_THREADS) {
        if (e.alive[base + p]) {
            const unsigned long long bits = dbl_bits(e.el[base + p]);
            lmin = min(lmin, bits); lmax = max(lmax, bits);
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        lmin = min(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    if ((threadIdx.x & 31) == 0) { s_min[threadIdx.x >> 5] = lmin; s_max[threadIdx.x >> 5] = lmax; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < STREAM_THREADS / 32; ++w) { lmin = min(lmin, s_min[w]); lmax = max(lmax, s_max[w]); }
        if (lmax >= lmin) { atomicMin(&s.min_el_bits, lmin); atomicMax(&s.max_el_bits, lmax); }
    }
    __syncthreads();
    }
}

// clear the z-buffer of the scans that re-project in full and fix their image geometry
__global__ void __launch_bounds__(STREAM_THREADS) k_clear_images(EngineDev e, int n_scans) {
    const int n_full = e.work_cnt[0];
    for (int li = blockIdx.y; li < n_full; li += gridDim.y) {
        const int b = e.full_list[li];
        ScanState& s = e.st[b];
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            e.far_arr[b] = 0;
            if (s.min_el_bits == R3D_EMPTY_U64) { set_error(s, R3D_ERR_ASSERT); }
            s.geom = make_geom(e.rows, e.cols, e.cols, bits_dbl(s.max_el_bits), bits_dbl(s.min_el_bits));
        }
        unsigned long long* z = e.zraw + (size_t)b * e.hw;
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < e.hw; i += gridDim.x * blockDim.x) z[i] = R3D_EMPTY_U64;
    }
}

// A3 (od/ins:85-130): bin every live point with the reference's truncation rule, write pix_id, 64-bit atomicMin of
// the range bits into the z-buffer.  Algorithmic traffic 20 B/point (+ 8 B/pixel for the z-buffer).
__global__ void __launch_bounds__(STREAM_THREADS) k_project(EngineDev e, int n_scans) {
    const int n_full = e.work_cnt[0];
    for (int li = blockIdx.y; li < n_full; li += gridDim.y) {
    const int b = e.full_list[li];
    ScanState& s = e.st[b];
    const int n = s.n0 + s.n_tail;
    const int p0 = blockIdx.x * CHUNK;
    if (p0 >= n) continue;
    const ImageGeom g = make_geom(e.rows, e.cols, e.cols, bits_dbl(s.max_el_bits), bits_dbl(s.min_el_bits));
    const size_t base = (size_t)b * e.P;           // P is a multiple of 16: the 4-point vectors below are aligned
    unsigned long long* z = e.zraw + (size_t)b * e.hw;
    auto one = [&](bool alive, double el, unsigned col, double r) -> int {
        if (!alive) return -1;
        const int row = bin_row(g, el);
        if (row < 0 || row >= g.rows) { set_error(s, R3D_ERR_ASSERT); return -1; }          // od/ins:111
        const int pix = row * g.cols + (int)col;
        atomicMin(&z[pix], dbl_bits(r));
        return pix;
    };
#pragma unroll 2
    for (int it = 0; it < CHUNK / (STREAM_THREADS * 4); ++it) {
        const int p = p0 + it * STREAM_THREADS * 4 + threadIdx.x * 4;
        if (p >= n) break;
        if (p + 3 < n) {                           // four points per thread: 4 + 32 + 8 + 32 bytes in, 16 out
            const uchar4 a = *reinterpret_cast<const uchar4*>(e.alive + base + p);
            if (!(a.x | a.y | a.z | a.w)) continue;
            const double2 e01 = *reinterpret_cast<const double2*>(e.el + base + p);
            const double2 e23 = *reinterpret_cast<const double2*>(e.el + base + p + 2);
            const ushort4 c = *reinterpret_cast<const ushort4*>(e.col + base + p);
            const double2 r01 = *reinterpret_cast<const double2*>(e.r + base + p);
            const double2 r23 = *reinterpret_cast<const double2*>(e.r + base + p + 2);
            int4 px;
            px.x = one(a.x, e01.x, c.x, r01.x); px.y = one(a.y, e01.y, c.y, r01.y);
            px.z = one(a.z, e23.x, c.z, r23.x); px.w = one(a.w, e23.y, c.w, r23.y);
            *reinterpret_cast<int4*>(e.pix + base + p) = px;
        } else {
            for (int q = p; q < n; ++q) e.pix[base + q] = one(e.alive[base + q], e.el[base + q], e.col[base + q], e.r[base + q]);
        }
    }
    }
}

struct RawImage {        // the engine's z-buffer as close/fill input
    const unsigned long long* raw;
    __device__ void load(int64_t i, double& v, uint8_t& o) const {
        const unsigned long long b = raw[i];
        const bool hit = b != R3D_EMPTY_U64;
        v = hit ? bits_dbl(b) : kEmptyRange;            // od/ins:100: empty = 500
        o = hit ? 3 : 0;
    }
    __device__ double lab(int64_t i) const { return raw[i] != R3D_EMPTY_U64 ? 1.0 : -1.0; }
};

// semseg addjust_map_2 (ss/ins:202-224): map cells (value != 0) that hold a live scene point with z < 1.5 and a
// non-ground label count as value 4 for this slot.  Kept as a per-scan bit window instead of rewriting the map.
// The reference indexes map[ix][iy] with the truncated world coordinates as they are: a negative index wraps around
// like any numpy index (cell size + ix), an index past the end raises IndexError (-> R3D_ERR_INDEX).  Wrapped cells
// lie far from the scan, outside the bit window: they go to a short per-scan list (occ_far).
// delta = 0: set the bit (full rebuild from the live points); +1 / -1: the point joined / left the scene — the per-cell
// COUNT of such points (occ_cnt) is kept, the bit follows count > 0 (incremental form used by the per-scan walker: the
// reference rebuilds the marks from the whole current scene at every slot, which is the same set of cells).
// `ignore_alive`: the caller knows the point qualifies as a scene point (it is being removed / was just appended).
__device__ __forceinline__ void adjust_map_point(const EngineDev& e, int b, ScanState& s, const double* T, int p, int delta,
                                                 bool ignore_alive) {
    const size_t base = (size_t)b * e.P;
    if (!ignore_alive && !e.alive[base + p]) return;
    const unsigned lab = e.label[base + p];
    bool ground = false;
    for (int i = 0; i < e.n_road_indexes; ++i) ground |= lab == (unsigned)e.road_indexes[i];
    if (ground) return;
    double x, y, z;
    load_xyz(e, b, p, s.n0, x, y, z);
    if (!(z < 1.5)) return;
    const double wx = add(add(add(mul(T[0], x), mul(T[1], y)), mul(T[2], z)), T[3]);
    const double wy = add(add(add(mul(T[4], x), mul(T[5], y)), mul(T[6], z)), T[7]);
    int ix = trunc_to_int(sub(wx, (double)e.ss_move_x));
    int iy = trunc_to_int(sub(wy, (double)e.ss_move_y));
    if (ix >= e.ss_sx || iy >= e.ss_sy || ix < -e.ss_sx || iy < -e.ss_sy) { if (delta >= 0) set_error(s, R3D_ERR_INDEX); return; }   // IndexError
    if (ix < 0) ix += e.ss_sx;                                   // numpy negative index
    if (iy < 0) iy += e.ss_sy;
    if (e.ss_map[(size_t)ix * e.ss_sy + iy] == 0) return;
    const int lx = ix - s.win_x0, ly = iy - s.win_y0;
    if (lx < 0 || ly < 0 || lx >= e.map_window || ly >= e.map_window) {
        if (delta < 0) return;                                   // far cells are not counted: the walker rebuilds in full when any exists
        int* far = e.occ_far + (size_t)b * (OCC_FAR_CAP + 1);        // small set: [0] = non-empty flag, then cells or -1
        const int cell = ix * e.ss_sy + iy;
        far[0] = 1;
        for (int i = 0; i < OCC_FAR_CAP; ++i) {
            const int old = atomicCAS(&far[1 + (cell + i) % OCC_FAR_CAP], -1, cell);
            if (old == -1 || old == cell) return;
        }
        set_error(s, R3D_ERR_CAPACITY);
        return;
    }
    const int bit = lx * e.map_window + ly;
    unsigned* word = &e.occ_win[(size_t)b * (e.map_window * e.map_window / 32) + (bit >> 5)];
    if (delta == 0) { atomicOr(word, 1u << (bit & 31)); return; }
    unsigned* cnt = &e.occ_cnt[(size_t)b * e.map_window * e.map_window + bit];
    if (delta > 0) { atomicAdd(cnt, 1u); atomicOr(word, 1u << (bit & 31)); }
    else if (atomicSub(cnt, 1u) == 1u) atomicAnd(word, ~(1u << (bit & 31)));
}

// count_too != 0: also build the per-cell counts (the walker keeps them up to date afterwards)
__global__ void __launch_bounds__(STREAM_THREADS) k_adjust_map(EngineDev e, int n_scans, int count_too = 0) {
    const int b = blockIdx.y;
    if (b >= n_scans || !e.gate_update[b]) return;
    ScanState& s = e.st[b];
    const int n = s.n0 + s.n_tail;
    const int p0 = blockIdx.x * CHUNK;
    if (p0 >= n) return;
    const double* T = e.poses + (size_t)b * 16;
    for (int p = p0 + threadIdx.x; p < min(p0 + CHUNK, n); p += STREAM_THREADS) adjust_map_point(e, b, s, T, p, count_too ? 1 : 0);
}
