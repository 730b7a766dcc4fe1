// Kernels of the batched Real3D-Aug engine, part: the per-scan persistent walker.
// Included by r3d_engine_kernels.cuh (inside namespace r3d, after the staged round kernels); not a standalone header.
// ------------------------------------------------------------------------------------------------ walker
// ONE CTA per scan runs the reference's whole per-scan `while` loop (od/ins:375-614, ss/ins:371-586) without returning
// to the host: scheduling step (A13) -> apply the last vis_px mask / refresh the range image around the inserted object
// (A11, A12, A3, A4) -> placement search of the next cut object (A5-A10) -> occlusion count (A11) -> selection and
// insertion (A12) -> next step.  Scans are independent (SURVEY 8e), so the CTAs never talk to each other: no
// co-residency requirement, no round barrier over the batch (the staged round kernels make every scan wait for the
// slowest one of every stage), no launch boundary between dependent stages, and the candidates of a try are visited
// in ORDERED WINDOWS with a real early exit at the first candidate that keeps min_points (od/ins:530-561).
// The once-per-scan streaming work (spherical ingest, indices, first full projection + close/fill, output
// compaction) stays in batch-wide HBM-bound kernels before / after this one.
// This header is included TWICE by r3d_engine_kernels.cuh, each time inside its own namespace and with its own CTA shape
// (R3D_WALK_THREADS x R3D_WALK_CTAS_PER_SM, both defined by the includer): `walk_od` = 384 threads x 3 CTAs per SM for
// the object-detection workloads (short tries: narrower CTAs leave fewer lanes idle at the barriers and the SM holds
// three scans; 256 x 3 gives +6 % more throughput but one batch alone takes 5.5 instead of 4.8 ms), `walk_ss` = 512 x 2
// for semseg (big objects: the map test / collision work of a try is throughput bound inside the CTA).
#ifdef R3D_WALK_NOINLINE
#define R3D_WALK_FN __noinline__
#else
#define R3D_WALK_FN
#endif
constexpr int WALK_THREADS = R3D_WALK_THREADS;
constexpr int WALK_CTAS_PER_SM = R3D_WALK_CTAS_PER_SM;
constexpr int WALK_W = WALK_THREADS / GRP;            // candidates per window = 8-lane groups of the CTA
constexpr int WALK_Q = WALK_W + WALK_THREADS / 32;    // candidate records: a window's worth + the leftover of a chunk (the OD queue)
constexpr int WALK_SEL_PTS = 1024;                    // object points / tile pixels the selection keeps in shared memory
#ifndef R3D_WALK_SEL_TILE
#define R3D_WALK_SEL_TILE 4096
#endif
constexpr int WALK_SEL_TILE = R3D_WALK_SEL_TILE;
constexpr int WALK_SEL_KEYS = 1024;                   // next_pow2(WALK_SEL_PTS)
constexpr int WALK_OCC_LANES = 64;                    // threads that count one feasible candidate's visible points
constexpr int WALK_OCC_PAR = WALK_THREADS / WALK_OCC_LANES;
constexpr int WALK_NWARPS = WALK_THREADS / 32;


// dynamic shared memory: [object x | y | z (fp64)] [ordered candidate list] [prefilter flags] [scratch]; the scratch
// holds the visible-pixel bit image of the exact occlusion count or the close/fill tile; the selection (after the
// last window of a try) reuses everything from offset 0
struct WalkSmem { size_t list_off, flags_off, scratch_off, total; };
__host__ __device__ __forceinline__ size_t walk_sel_bytes() {
    return (size_t)WALK_SEL_KEYS * 8 + (size_t)WALK_SEL_PTS * 8 + (size_t)WALK_SEL_TILE * 8 + (size_t)WALK_SEL_PTS * 4 +
           2 * (size_t)(WALK_SEL_TILE / 32) * 4 + 16;
}
__host__ __device__ __forceinline__ WalkSmem walk_smem_layout(int K, int dwords) {
    WalkSmem L;
    size_t o = (size_t)3 * OBJ_SMEM_PTS * 8;
    L.list_off = o; o += ((size_t)(K + 1) * 2 + 15) & ~(size_t)15;
    L.flags_off = o; o += ((size_t)(K + 1) + 15) & ~(size_t)15;
    L.scratch_off = o;
    const size_t occ = (size_t)dwords * 4;
    const size_t cf = (size_t)CF_SH * CF_SW * 8 + 4 * (size_t)CF_SH * CF_WORDS * 4;
    o += occ > cf ? occ : cf;
    const size_t sel = walk_sel_bytes();
    L.total = o > sel ? o : sel;
    if (L.total < sizeof(CfPipeSmem)) L.total = sizeof(CfPipeSmem);
    return L;
}

// phase clocks (SM cycles, summed over all scans by thread 0 of each CTA) -> e.stats[WALK_T0 + phase]
enum : int { WT_CTRL = 0, WT_UPDATE, WT_SETUP, WT_PLACE, WT_OCCL, WT_SELECT, WT_TOTAL, WT_ONMAP, WT_LEVEL_WARP, WT_COLLIDE_WARP,
              WT_N_LEVEL, WT_N_COLLIDE, WT_APPLY, WT_PATCH, WT_CLOSEFILL, WT_SS_RESWEEP, WT_SS_LEVEL, WT_COUNT };
constexpr int WALK_T0 = 16;
struct WalkClock {
    long long t;
    __device__ __forceinline__ void start() { if (threadIdx.x == 0) t = clock64(); }
    __device__ __forceinline__ void lap(const EngineDev& e, int phase) {
        if (threadIdx.x == 0) { const long long n = clock64(); atomicAdd(&e.stats[WALK_T0 + phase], (unsigned long long)(n - t)); t = n; }
    }
};

struct WalkCtl {                 // control block of the CTA (static shared memory)
    int apply, project, tryact;
    int n_list, nfw, n_feas, found;
    int found_k, last_k;
    double found_level, last_level;
    double dz_run, dz_next;      // semseg: the z shift carried from yaw to yaw (ss/fs:146-147)
    int changed;
    int cnt_lo[WALK_OCC_PAR], cnt_hi[WALK_OCC_PAR];
    int exact_cnt;
    int wk[WALK_Q];              // rotation of the candidates (semseg: a window's; OD: the ring of on-map candidates)
    unsigned char wflag[WALK_Q];
    double wlevel[WALK_Q];
    int wfeas[WALK_W];           // window-local indices of the feasible candidates, in rotation order
    int won[WALK_W];             // window-local indices of the candidates the next sub-stage works on
    int wsub[WALK_W];            // chunk-local list (candidates of the chunk that have a road level)
    int n_sub;
    int next;                    // dynamic task counter of a sub-stage
    double wcx[WALK_Q], wcy[WALK_Q];     // centre of the candidates (the box centre turned about the sensor)
    int a_k[WALK_W];             // OD stage A (map test) of a window, before the on-map ones join the queue
    unsigned char a_on[WALK_W];
    double a_cx[WALK_W], a_cy[WALK_W];
    int wlist[WALK_THREADS / 32];        // records of the chunk being worked on (OD)
    unsigned surf[R3D_MAX_SURFACE];      // labels the tried class may stand on (road-level search)
    int n_surf;
    double wdz[WALK_W];          // semseg fixed point: the shift candidate i was (or must be) tested under
    double wtol[WALK_W];         // ... and how far the shift may move from it without changing the verdict of the map test
    unsigned long long wtolp[WALK_W], wtolb[WALK_W];   // its parts while the map test runs: min over on-map points, max over off-map points
    int wbad[WALK_W];
    int whit[WALK_Q];            // collision found by one of the warps that share a candidate
    int witness;                 // original point that made an earlier candidate of the try collide (-1: none yet)
    unsigned char wpass[WALK_W], wtodo[WALK_W], whok[WALK_W], whas[WALK_W];
    ObjBox ob;
    int s_warp[WALK_NWARPS];
    int upd_full, upd_patch, rect[4];
    unsigned long long el_min, el_max;
    __align__(16) float wclip[WALK_NWARPS][8];     // per warp: column bounds of the collision walk over a long box (make_row_clip)
};

// ---- A4 on a pixel rectangle, any CTA size (the batch-wide kernel is r3d_closefill.cuh): tiles of CF_TH x CF_TW
// outputs staged with their halo in shared memory, bit-row morphology, ordered fp64 neighbour mean
__device__ R3D_WALK_FN void walk_close_fill(const EngineDev& e, int b, const int* rect, unsigned char* scratch) {
    unsigned long long (*s_raw)[CF_SW] = reinterpret_cast<unsigned long long (*)[CF_SW]>(scratch);
    unsigned (*s_one)[CF_WORDS] = reinterpret_cast<unsigned (*)[CF_WORDS]>(scratch + (size_t)CF_SH * CF_SW * 8);
    unsigned (*s_in)[CF_WORDS] = s_one + CF_SH;
    unsigned (*s_dil)[CF_WORDS] = s_in + CF_SH;
    unsigned (*s_ero)[CF_WORDS] = s_dil + CF_SH;
    const int H = e.rows, W = e.cols, tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    const unsigned long long* raw = e.zraw + (size_t)b * e.hw;
    double* out = e.smooth + (size_t)b * e.hw;
    auto left = [](const unsigned* a, int w) { return (a[w] << 1) | (w > 0 ? a[w - 1] >> 31 : 0u); };
    auto right = [](const unsigned* a, int w) { return (a[w] >> 1) | (a[w + 1] << 31); };
    bool far = false;
    for (int r0 = rect[0]; r0 <= rect[1]; r0 += CF_TH)
        for (int c0 = rect[2]; c0 <= rect[3]; c0 += CF_TW) {
            // only the rows / columns of the rectangle (+ halo) are staged and computed: a typical object covers a few
            // hundred pixels, not a whole 32 x 64 tile
            const int th = min(CF_TH, rect[1] - r0 + 1), tw = min(CF_TW, rect[3] - c0 + 1);
            const int sh = th + 2 * CF_HR, sw = tw + 2 * CF_HC;
            for (int i = tid; i < sh * sw; i += nt) {
                const int lr = i / sw, lc = i % sw;
                const int r = r0 - CF_HR + lr, c = c0 - CF_HC + lc;
                s_raw[lr][lc] = (r >= 0 && r < H && c >= 0 && c < W) ? raw[(size_t)r * W + c] : R3D_EMPTY_U64;
            }
            if (tid < sh) { s_one[tid][3] = 0u; s_in[tid][3] = 0u; s_dil[tid][3] = ~0u; }
            __syncthreads();
            for (int u = warp; u < sh * 3; u += nwarps) {             // bit rows of the staged tile
                const int lr = u / 3, w = u % 3, lc = w * 32 + lane;
                const int r = r0 - CF_HR + lr, c = c0 - CF_HC + lc;
                const bool inside = lc < sw && r >= 0 && r < H && c >= 0 && c < W;
                const bool hit = inside && s_raw[lr][min(lc, sw - 1)] != R3D_EMPTY_U64;
                const unsigned b_one = __ballot_sync(0xffffffffu, hit), b_in = __ballot_sync(0xffffffffu, inside);
                if (lane == 0) { s_one[lr][w] = b_one; s_in[lr][w] = b_in; }
            }
            __syncthreads();
            for (int t = tid; t < (sh - 4) * 3; t += nt) {
                const int lr = 2 + t / 3, w = t % 3;
                unsigned d = 0u;
#pragma unroll
                for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = s_one[lr + dr]; d |= a[w] | left(a, w) | right(a, w); }
                s_dil[lr][w] = d | ~s_in[lr][w];
            }
            __syncthreads();
            for (int t = tid; t < th * 3; t += nt) {
                const int lr = CF_HR + t / 3, w = t % 3;
                unsigned er = ~0u;
#pragma unroll
                for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = s_dil[lr + dr]; er &= a[w] & left(a, w) & right(a, w); }
                s_ero[lr][w] = er;
            }
            __syncthreads();
            for (int i = tid; i < th * tw; i += nt) {
                const int lr = i / tw, lc = i % tw;
                const int r = r0 + lr, c = c0 + lc;
                if (r >= H || c >= W) continue;
                const int sr = lr + CF_HR, sc = lc + CF_HC;
                const bool er = (s_ero[sr][sc >> 5] >> (sc & 31)) & 1u;
                const bool one = (s_one[sr][sc >> 5] >> (sc & 31)) & 1u;
                double tv = one ? bits_dbl(s_raw[sr][sc]) : kEmptyRange;          // od/ins:100: empty = 500
                if (er && !one) {                                                // cl:41-43
                    int neighbors = 0;
                    double sum = 0.0;
                    const int q = sc - 1, qw = q >> 5, qb = q & 31;
#pragma unroll
                    for (int dr = -2; dr <= 2; ++dr) {                           // cl:46-51, (drow, dcol) order
                        const unsigned m = __funnelshift_r(s_one[sr + dr][qw], s_one[sr + dr][qw + 1], qb) & 7u;
                        if (m & 1u) { neighbors += 1; sum = add(sum, bits_dbl(s_raw[sr + dr][sc - 1])); }
                        if (m & 2u) { neighbors += 1; sum = add(sum, bits_dbl(s_raw[sr + dr][sc])); }
                        if (m & 4u) { neighbors += 1; sum = add(sum, bits_dbl(s_raw[sr + dr][sc + 1])); }
                    }
                    if (neighbors > 0) tv = mean_div(sum, neighbors);   // cl:57
                }
                out[(size_t)r * W + c] = tv;
                far |= tv > kEmptyRange;
            }
            __syncthreads();                                  // the tile buffers are reused by the next tile
        }
    if (far) atomicOr(&e.far_arr[b], 1);
}

// ---- A2 + A3 for the whole scan inside the CTA: the rare slot whose elevation range moved (the first projection of
// every scan is done batch-wide by k_minmax / k_clear_images / k_project before the walker starts)
__device__ R3D_WALK_FN void walk_full_reproject(const EngineDev& e, int b, ScanState& s, WalkCtl& c) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const size_t base = (size_t)b * e.P;                 // rows are padded to a multiple of 16 points: 4-point vectors
    const int n = s.n0 + s.n_tail, n4 = (n + 3) >> 2;
    const unsigned* __restrict__ alive4 = reinterpret_cast<const unsigned*>(e.alive + base);
    const double2* __restrict__ el2 = reinterpret_cast<const double2*>(e.el + base);
    if (tid == 0) { c.el_min = R3D_EMPTY_U64; c.el_max = 0ull; }
    unsigned long long* z = e.zraw + (size_t)b * e.hw;
    if ((reinterpret_cast<size_t>(z) & 15) == 0) {
        ulonglong2* z2 = reinterpret_cast<ulonglong2*>(z);
        for (int i = tid; i < e.hw / 2; i += nt) z2[i] = make_ulonglong2(R3D_EMPTY_U64, R3D_EMPTY_U64);
        if ((e.hw & 1) && tid == 0) z[e.hw - 1] = R3D_EMPTY_U64;
    } else {                                             // odd image size: the scan's z-buffer starts on an 8-byte boundary
        for (int i = tid; i < e.hw; i += nt) z[i] = R3D_EMPTY_U64;
    }
    __syncthreads();
    unsigned long long lmin = R3D_EMPTY_U64, lmax = 0ull;
#pragma unroll 2
    for (int q = tid; q < n4; q += nt) {
        const unsigned a = alive4[q];
        if (!a) continue;
        const double2 lo = el2[2 * q], hi = el2[2 * q + 1];
        const double ev[4] = {lo.x, lo.y, hi.x, hi.y};
#pragma unroll
        for (int u = 0; u < 4; ++u)
            if (((a >> (8 * u)) & 0xFFu) && 4 * q + u < n) { const unsigned long long bits = dbl_bits(ev[u]); lmin = min(lmin, bits); lmax = max(lmax, bits); }
    }
    for (int o = 16; o > 0; o >>= 1) {
        lmin = min(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    if ((tid & 31) == 0 && lmax >= lmin) { atomicMin(&c.el_min, lmin); atomicMax(&c.el_max, lmax); }
    __syncthreads();
    const unsigned long long mn = c.el_min, mx = c.el_max;
    if (tid == 0) {
        s.min_el_bits = mn; s.max_el_bits = mx;
        e.far_arr[b] = 0;
        if (mn == R3D_EMPTY_U64) set_error(s, R3D_ERR_ASSERT);
        s.geom = make_geom(e.rows, e.cols, e.cols, bits_dbl(mx), bits_dbl(mn));
        atomicAdd(&e.stats[11], 1ull);
    }
    const ImageGeom g = make_geom(e.rows, e.cols, e.cols, bits_dbl(mx), bits_dbl(mn));
    const double2* __restrict__ r2 = reinterpret_cast<const double2*>(e.r + base);
    const ushort4* __restrict__ col4 = reinterpret_cast<const ushort4*>(e.col + base);
    int4* pix4 = reinterpret_cast<int4*>(e.pix + base);
#pragma unroll 2
    for (int q = tid; q < n4; q += nt) {
        const unsigned a = alive4[q];
        int px[4] = {-1, -1, -1, -1};
        if (a) {
            const double2 lo = el2[2 * q], hi = el2[2 * q + 1], rl = r2[2 * q], rh = r2[2 * q + 1];
            const ushort4 cc = col4[q];
            const double ev[4] = {lo.x, lo.y, hi.x, hi.y}, rv[4] = {rl.x, rl.y, rh.x, rh.y};
            const int cv[4] = {cc.x, cc.y, cc.z, cc.w};
#pragma unroll
            for (int u = 0; u < 4; ++u)
                if (((a >> (8 * u)) & 0xFFu) && 4 * q + u < n) {
                    const int row = bin_row(g, ev[u]);
                    if (row < 0 || row >= g.rows) set_error(s, R3D_ERR_ASSERT);                  // od/ins:111
                    else { px[u] = row * g.cols + cv[u]; atomicMin(&z[px[u]], dbl_bits(rv[u])); }
                }
        }
        pix4[q] = make_int4(px[0], px[1], px[2], px[3]);
    }
}

// ---- semseg addjust_map_2 (ss/ins:202-224) for the scan's live points (same rule as k_adjust_map)
__device__ R3D_WALK_FN void walk_adjust_map(const EngineDev& e, int b, ScanState& s) {
    const int n = s.n0 + s.n_tail;
    const double* T = e.poses + (size_t)b * 16;
    for (int p = threadIdx.x; p < n; p += blockDim.x) adjust_map_point(e, b, s, T, p);
}

// ---- slot update: what k_update + the refresh kernels of a staged round do for one scan
__device__ R3D_WALK_FN void walk_update(const EngineDev& e, int b, ScanState& s, WalkCtl& c, int do_apply, int do_update,
                            unsigned char* scratch, unsigned char* dyn) {
    long long ut = clock64();
    auto ulap = [&](int phase) {
        if (threadIdx.x == 0) { const long long n = clock64(); atomicAdd(&e.stats[WALK_T0 + phase], (unsigned long long)(n - ut)); ut = n; }
    };
    const int tid = threadIdx.x, nt = blockDim.x;
    const size_t base = (size_t)b * e.P;
    const bool ext = do_apply && (e.task == 1 ? apply_vis_mask<true>(e, b, s, tid, nt) : apply_vis_mask<false>(e, b, s, tid, nt));
    const int extreme = __syncthreads_or(ext);
    ulap(WT_APPLY);
    if (tid == 0) {
        int full = 0, patch = 0;
        int* rect = c.rect;
        rect[0] = 0; rect[1] = -1; rect[2] = 0; rect[3] = -1;
        if (do_update) {
            const bool extended = s.new_min_bits < s.min_el_bits || s.new_max_bits > s.max_el_bits;
            full = s.first || extreme || extended || e.far_arr[b] || e.force_full;
            patch = !full;
            if (full) {
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
        c.upd_full = full; c.upd_patch = patch;
    }
    __syncthreads();
    // semseg map marks (addjust_map_2): kept incrementally by the removals above and the insertions of walk_try; a
    // scan with marked cells outside the bit window (numpy-wrapped indices) rebuilds them from all its live points
    const bool rebuild_marks = do_update && e.task == 1 && s.far_flag;
    if (rebuild_marks) {
        const int ww = e.map_window * e.map_window / 32;
        unsigned* o = e.occ_win + (size_t)b * ww;
        for (int i = tid; i < ww; i += nt) o[i] = 0u;
        occ_far_clear(e, b, tid);
        __syncthreads();
    }
    if (c.upd_patch) {
        unsigned long long* z = e.zraw + (size_t)b * e.hw;
        const unsigned* dm = e.dmask + (size_t)b * e.dwords;
        if (s.d_r1 >= s.d_r0 && s.d_c1 >= s.d_c0) {
            const int nw = (s.d_c1 >> 5) - (s.d_c0 >> 5) + 2, nrow = s.d_r1 - s.d_r0 + 1;
            for (int i = tid; i < nrow * nw; i += nt) {
                const int r = s.d_r0 + i / nw;
                const int w = ((r * e.cols + s.d_c0) >> 5) + i % nw;
                if (w > ((r * e.cols + s.d_c1) >> 5)) continue;
                unsigned m = dm[w];
                while (m) { const int bit = __ffs(m) - 1; m &= m - 1; z[(w << 5) + bit] = R3D_EMPTY_U64; }
            }
        }
        __syncthreads();
        if (s.apply_flag)                                        // points appended by the accept being applied
            for (int p = s.n0 + s.tail_before + tid; p < s.n0 + s.n_tail; p += nt)
                if (e.alive[base + p]) atomicMin(&z[e.pix[base + p]], dbl_bits(e.r[base + p]));
    } else if (c.upd_full) {
        walk_full_reproject(e, b, s, c);
    }
    __syncthreads();
    ulap(WT_PATCH);
    if (c.upd_full && !(e.cols & 1)) {
        // the whole image: the tiles stream through two shared-memory buffers (cp.async), as in the batch-wide kernel;
        // the object staging area of the dynamic shared memory is free between two tries
        const int tiles = e.cf_tiles;
        cf_pipelined_tiles<WALK_THREADS>(*reinterpret_cast<CfPipeSmem*>(dyn), e.zraw, e.rows, e.cols, (int64_t)e.hw, e.smooth, e.far_arr,
                                         0, tiles, 1, [&](int t) { return b * tiles + t; });
    } else if (c.rect[1] >= c.rect[0] && c.rect[3] >= c.rect[2]) walk_close_fill(e, b, c.rect, scratch);
    ulap(WT_CLOSEFILL);
    if (rebuild_marks) { __syncthreads(); walk_adjust_map(e, b, s); }
    __syncthreads();
}

// ---- ordered list of the window entries i < nw with pred(i) -> out[]; every thread calls it (two barriers); also
// re-arms the dynamic task counter of the next sub-stage
template <class P>
__device__ __forceinline__ int walk_window_list(WalkCtl& c, int nw, int* out, P pred) {
    const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
    constexpr int NWW = (WALK_W + 31) / 32;
    bool on = false;
    unsigned m = 0u;
    if (w < NWW) {
        on = tid < nw && pred(tid);
        m = __ballot_sync(0xffffffffu, on);
        if (lane == 0) c.s_warp[w] = __popc(m);
    }
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int i = 0; i < NWW; ++i) { if (i < w) off += c.s_warp[i]; tot += c.s_warp[i]; }
    if (on) out[off + __popc(m & ((1u << lane) - 1u))] = tid;
    if (tid == 0) c.next = 0;
    __syncthreads();
    return tot;
}

// ---- A5 + A6a (od/fs:263-279) on EVERY object point for one yaw candidate, one 8-lane group
__device__ __forceinline__ bool walk_onmap_od(const EngineDev& e, int b, const ObjBox& ob, const ClassCfg& cc, const double* ox,
                                              const double* oy, int k, int gl, unsigned gm) {
    const int count = ob.count, msel = cc.map_sel;
    const int* dims = e.od_map_dims + ((size_t)b * 2 + msel) * 4;
    const int sx = dims[0], sy = dims[1];
    const double mx = (double)dims[2], my = (double)dims[3];
    const unsigned char* map = e.od_maps + e.od_map_off[(size_t)b * 2 + msel];
    const double c = e.cos_k[k], sn = e.sin_k[k];
    bool any_in = false, bad = false;
    for (int i0 = 0; i0 < count; i0 += 4 * GRP) {
        double x[4], y[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = min(i0 + u * GRP + gl, count - 1);           // the clamped repeats change nothing
            x[u] = ox[i]; y[u] = oy[i];
        }
        unsigned char v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            v[u] = 1;
            const double gx = sub(sub(mul(c, x[u]), mul(sn, y[u])), mx), gy = sub(add(mul(sn, x[u]), mul(c, y[u])), my);
            if (!(gx < 0.0 || gx >= (double)sx || gy < 0.0 || gy >= (double)sy)) {
                any_in = true; v[u] = __ldg(&map[(size_t)((int)gx) * sy + (int)gy]);
            }
        }
        bad = v[0] != 1 || v[1] != 1 || v[2] != 1 || v[3] != 1;
        if (__ballot_sync(gm, bad) & gm) { bad = true; break; }       // od/fs:277-279
    }
    return (__ballot_sync(gm, any_in) & gm) != 0u && !bad;
}

// ---- A7 for the window candidates listed in c.won[0 .. n): ONE WARP per candidate, dealt dynamically (a free warp takes
// the next one): the ring search is a chain of dependent cell / point loads, 32 lanes keep four rows of cells in flight
__device__ R3D_WALK_FN void walk_levels(const EngineDev& e, int b, WalkCtl& c, const int* list, int n) {
    const int lane = threadIdx.x & 31;
    for (;;) {
        int t = 0;
        if (lane == 0) t = atomicAdd(&c.next, 1);
        t = __shfl_sync(0xffffffffu, t, 0);
        if (t >= n) break;
        const int i = list[t];
        double level = 0.0;
        const long long t0 = clock64();
        const bool ok = e.task == 0 ? warp_road_level<false>(e, b, c.surf, c.n_surf, c.wcx[i], c.wcy[i], lane, level)
                                    : warp_road_level<true>(e, b, c.surf, c.n_surf, c.wcx[i], c.wcy[i], lane, level);
        if (lane == 0) {
            c.wflag[i] = (unsigned char)(ok ? (CF_ONMAP | CF_HOK) : CF_ONMAP);           // od/fs:281-285
            c.wlevel[i] = level;
            atomicAdd(&e.stats[WALK_T0 + WT_LEVEL_WARP], (unsigned long long)(clock64() - t0)); atomicAdd(&e.stats[WALK_T0 + WT_N_LEVEL], 1ull);
        }
    }
}

// ---- A8 + A9 for the window candidates listed in c.won[0 .. n) (they have a road level), one warp per candidate
__device__ R3D_WALK_FN void walk_collides(const EngineDev& e, int b, const ScanState& s, WalkCtl& c, const int* list, int n) {
    // n <= WALK_NWARPS candidates (a chunk): the warps are dealt statically, and when the chunk is short the spare warps
    // join in — `wpc` warps per candidate share its obstacle-grid rows (semseg chunks hold ~6 candidates whose boxes cover
    // thousands of grid points each)
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const ObjBox& ob = c.ob;
    const ClassCfg& cc = e.classes[ob.cls];
    if (n <= 0) return;
    const int wpc = max(1, WALK_NWARPS / n);
    const int t = warp / wpc, part = warp % wpc;
    if (t >= n) return;
    const int i = list[t], k = c.wk[i];
    const long long t0 = clock64();
    const bool hit = warp_collides(e, b, s, ob, cc, e.cos_k[k], e.sin_k[k], c.wlevel[i], lane, part, wpc, &c.whit[i], &c.witness,
                                   c.wclip[warp]);
    if (lane == 0) {
        if (hit && atomicExch(&c.whit[i], 1) == 0) c.wflag[i] = (unsigned char)(CF_ONMAP | CF_HOK | CF_COLLIDE);   // the first of the warps that share it
        if (part == 0) { atomicAdd(&e.stats[WALK_T0 + WT_COLLIDE_WARP], (unsigned long long)(clock64() - t0)); atomicAdd(&e.stats[WALK_T0 + WT_N_COLLIDE], 1ull); }
    }
}

// ---- semseg window: A6b with the carried z shift as a fixed-point iteration over the window's yaws (see k_onmap_ss),
// the road level searched only for the yaws that pass the map test, then A8/A9
__device__ R3D_WALK_FN int walk_window_ss(const EngineDev& e, int b, ScanState& s, WalkCtl& c, const double* ox, const double* oy,
                              const double* oz, int base, int nw) {
    const int tid = threadIdx.x, g = tid / GRP, gl = tid % GRP;
    const unsigned gm = group_mask();
    const ObjBox& ob = c.ob;
    const ClassCfg& cc = e.classes[ob.cls];
    if (tid < nw) {
        const int kk = base + tid + 1;
        const double ck = e.cos_k[kk], sk = e.sin_k[kk];
        c.wk[tid] = kk; c.wdz[tid] = c.dz_run; c.wpass[tid] = 0; c.wtodo[tid] = 1; c.whas[tid] = 0; c.whok[tid] = 0;
        c.wlevel[tid] = 0.0; c.wflag[tid] = 0; c.won[tid] = tid;
        c.wcx[tid] = sub(mul(ck, c.ob.cx), mul(sk, c.ob.cy)); c.wcy[tid] = add(mul(sk, c.ob.cx), mul(ck, c.ob.cy));
    }
    __syncthreads();
    const double* T = e.poses + (size_t)b * 16;
    SsMapTest m;
    m.t00 = T[0]; m.t01 = T[1]; m.t02 = T[2]; m.t03 = T[3]; m.t10 = T[4]; m.t11 = T[5]; m.t12 = T[6]; m.t13 = T[7];
    m.okmask = cc.map_ok_mask;
    m.occ = e.occ_win + (size_t)b * (e.map_window * e.map_window / 32);
    m.far = e.occ_far + (size_t)b * (OCC_FAR_CAP + 1);
    m.inv02 = m.t02 != 0.0 ? 1.0 / fabs(m.t02) : 1e300;
    m.inv12 = m.t12 != 0.0 ? 1.0 / fabs(m.t12) : 1e300;
    const int k = base + g + 1;
    const double cs = g < nw ? e.cos_k[k] : 1.0, sn = g < nw ? e.sin_k[k] : 0.0;
    const int warp = tid >> 5, lane = tid & 31;
    constexpr int ITEM_PTS = 128;                                 // object points per work item of the full map test
    const int n_items_per = ob.count > 4 * GRP ? (ob.count - 4 * GRP + ITEM_PTS - 1) / ITEM_PTS : 0;
    for (int sweep = 0; sweep <= nw; ++sweep) {
        long long t_ph = clock64();
        // (1) ss/fs:231-248 under the assumed shift, first on the first 32 object points (an 8-lane group per yaw: most
        // off-map yaws end here).  tolerated change of the shift: a yaw that passes keeps its verdict while EVERY point
        // keeps its map cell, a yaw that fails while ONE of its off-map points does
        if (g < nw && c.wtodo[g]) {
            const double dz = c.wdz[g];
            bool off = false;
            double tol_pass = 1e300, tol_bad = 0.0;
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int i = min(u * GRP + gl, ob.count - 1);                          // the clamped repeats change nothing
                double tol;
                const bool o = ss_point_off_map_t<true>(e, s, m, ox[i], oy[i], oz[i], cs, sn, dz, tol);
                tol = fmax(tol, 0.0);
                off |= o;
                if (o) tol_bad = fmax(tol_bad, tol); else tol_pass = fmin(tol_pass, tol);
            }
            const bool bad = (__ballot_sync(gm, off) & gm) != 0u;
            double tol = bad ? tol_bad : tol_pass;
#pragma unroll
            for (int o = GRP / 2; o > 0; o >>= 1) {
                const double other = __shfl_xor_sync(gm, tol, o);
                tol = bad ? fmax(tol, other) : fmin(tol, other);
            }
            if (gl == 0) {
                c.wbad[g] = bad ? 1 : 0;
                c.wtolp[g] = dbl_bits(bad ? 1e300 : tol); c.wtolb[g] = dbl_bits(bad ? tol : 0.0);
            }
        }
        __syncthreads();
        // (2) the rest of the points of the yaws that are still on the map: (yaw, 128-point chunk) items dealt to the warps
        // of the whole CTA (a big object on a few surviving yaws would otherwise keep 8 lanes busy and 500 waiting)
        const int n_live = n_items_per ? walk_window_list(c, nw, c.wsub, [&](int i) { return c.wtodo[i] && !c.wbad[i]; }) : 0;
        for (int t = warp; t < n_live * n_items_per; t += WALK_NWARPS) {
            const int i = c.wsub[t / n_items_per], q = t % n_items_per;
            if (*(volatile int*)&c.wbad[i]) continue;                                   // another chunk already found an off-map point
            const int kk = base + i + 1;
            const double ci = e.cos_k[kk], si = e.sin_k[kk], dz = c.wdz[i];
            bool off = false;
            double tol_pass = 1e300, tol_bad = 0.0;
#pragma unroll
            for (int u = 0; u < ITEM_PTS / 32; ++u) {
                const int p = 4 * GRP + q * ITEM_PTS + u * 32 + lane;
                if (p < ob.count) {
                    double tol;
                    const bool o = ss_point_off_map_t<true>(e, s, m, ox[p], oy[p], oz[p], ci, si, dz, tol);
                    tol = fmax(tol, 0.0);
                    off |= o;
                    if (o) tol_bad = fmax(tol_bad, tol); else tol_pass = fmin(tol_pass, tol);
                }
            }
            const bool bad = __any_sync(0xffffffffu, off);
            double tol = bad ? tol_bad : tol_pass;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double other = __shfl_xor_sync(0xffffffffu, tol, o);
                tol = bad ? fmax(tol, other) : fmin(tol, other);
            }
            if (lane == 0) {
                if (bad) { atomicMax(&c.wtolb[i], dbl_bits(tol)); atomicExch(&c.wbad[i], 1); }
                else atomicMin(&c.wtolp[i], dbl_bits(tol));
            }
        }
        __syncthreads();
        if (tid < nw && c.wtodo[tid]) {
            const bool bad = c.wbad[tid] != 0;
            c.wpass[tid] = bad ? 0 : 1;
            c.wtol[tid] = bits_dbl(bad ? c.wtolb[tid] : c.wtolp[tid]);
        }
        __syncthreads();
        if (tid == 0) { const long long n = clock64(); atomicAdd(&e.stats[WALK_T0 + WT_ONMAP], (unsigned long long)(n - t_ph)); t_ph = n; }
        // (3) ss/fs:250: correct_height of the yaws on the map that have no road level yet, one warp per yaw
        const int n_lvl = walk_window_list(c, nw, c.wsub, [&](int i) { return c.wpass[i] && !c.whas[i]; });
        walk_levels(e, b, c, c.wsub, n_lvl);
        __syncthreads();
        if (tid < n_lvl) {
            const int i = c.wsub[tid];
            c.whas[i] = 1; c.whok[i] = (c.wflag[i] & CF_HOK) ? 1 : 0;
        }
        __syncthreads();
        if (tid == 0) {                                           // the ordered walk over the flags (ss/fs:144-148)
            const long long n = clock64(); atomicAdd(&e.stats[WALK_T0 + WT_SS_LEVEL], (unsigned long long)(n - t_ph));
            double run = c.dz_run;
            int changed = 0;
            for (int i = 0; i < nw; ++i) {
                // yaw i was tested under another shift: test it again unless the shift stayed within the interval in
                // which none of the deciding points can change its map cell
                const bool redo = run != c.wdz[i] && !(fabs(run - c.wdz[i]) < c.wtol[i]);
                c.wtodo[i] = redo;
                if (redo) { c.wdz[i] = run; changed = 1; }
                if (c.wpass[i] && c.whok[i]) run = sub(c.wlevel[i], ob.cz);
            }
            c.changed = changed; c.dz_next = run;
            if (changed) atomicAdd(&e.stats[WALK_T0 + WT_SS_RESWEEP], 1ull);
        }
        __syncthreads();
        if (!c.changed) break;
    }
    if (tid < nw) c.wflag[tid] = c.wpass[tid] ? (c.whok[tid] ? (CF_ONMAP | CF_HOK) : CF_ONMAP) : 0;
    if (tid == 0) c.dz_run = c.dz_next;
    return walk_window_list(c, nw, c.won, [&](int i) { return c.wpass[i] && c.whok[i]; });
}

// ---- exact A11 count of one candidate with the whole CTA (visible-pixel bit image in shared memory), for the
// candidates the two-sided bound of walk_try cannot decide
__device__ R3D_WALK_FN int walk_exact_visible(const EngineDev& e, int b, ScanState& s, WalkCtl& c, int k, double level, unsigned* bits) {
    const int tid = threadIdx.x, nt = blockDim.x;
    const ObjBox& ob = c.ob;
    const ImageGeom g = s.geom;
    const double* smooth = e.smooth + (size_t)b * e.hw;
    int* pixbuf = e.occ_pix + (size_t)b * OCC_G * e.max_obj_points;
    for (int i = tid; i < e.dwords; i += nt) bits[i] = 0u;
    if (tid == 0) { c.exact_cnt = 0; atomicAdd(&e.stats[10], 1ull); }
    __syncthreads();
    const double cs = e.cos_k[k], sn = e.sin_k[k], dz = sub(level, ob.cz);
    const FastGeom fg = make_fast_geom(g);
    for (int i = tid; i < ob.count; i += nt) {
        const ObjPix o = project_obj_pix(e, ob, g, fg, i, cs, sn, dz, s);
        pixbuf[i] = o.pix;
        if (o.pix >= 0 && o.r < smooth[o.pix]) atomicOr(&bits[o.pix >> 5], 1u << (o.pix & 31));
    }
    __syncthreads();
    int cnt = 0;
    for (int i = tid; i < ob.count; i += nt) {
        const int pix = pixbuf[i];
        if (pix >= 0 && (bits[pix >> 5] & (1u << (pix & 31)))) ++cnt;
    }
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((tid & 31) == 0 && cnt) atomicAdd(&c.exact_cnt, cnt);
    __syncthreads();
    const int v = c.exact_cnt;
    __syncthreads();
    return v;
}

// ---- one tried cut object (od/ins:430-561)
__device__ R3D_WALK_FN void walk_try(const EngineDev& e, int b, ScanState& s, WalkCtl& c, unsigned char* dyn, const WalkSmem& L, WalkClock& clk) {
    const int K = e.K, tid = threadIdx.x, nt = blockDim.x;
    double* s_ox = reinterpret_cast<double*>(dyn);
    double* s_oy = s_ox + OBJ_SMEM_PTS;
    double* s_oz = s_oy + OBJ_SMEM_PTS;
    unsigned short* s_list = reinterpret_cast<unsigned short*>(dyn + L.list_off);
    unsigned char* s_flags = dyn + L.flags_off;
    unsigned char* scratch = dyn + L.scratch_off;
    if (tid == 0) {
        c.ob = e.obj[s.cur_obj];
        e.try_obj[b] = c.ob;
        c.n_feas = 0; c.found = -1; c.last_k = 0; c.last_level = 0.0; c.dz_run = 0.0; c.witness = -1;
        const ClassCfg& tc = e.classes[c.ob.cls];
        c.n_surf = tc.n_surface;
        for (int i = 0; i < R3D_MAX_SURFACE; ++i) c.surf[i] = i < tc.n_surface ? (unsigned)tc.surface[i] : 0xFFFFFFFFu;
        atomicAdd(&e.stats[1], 1ull);
    }
    __syncthreads();
    const ObjBox& ob = c.ob;
    const ClassCfg& cc = e.classes[ob.cls];
    const double *ox = e.obj_x + ob.first, *oy = e.obj_y + ob.first, *oz = e.obj_z + ob.first;
    if (ob.count <= OBJ_SMEM_PTS) {
        for (int i = tid; i < ob.count; i += nt) { s_ox[i] = ox[i]; s_oy[i] = oy[i]; s_oz[i] = oz[i]; }
        ox = s_ox; oy = s_oy; oz = s_oz;
    }
    int n_list = K;
    if (e.task == 0) {                   // A5 + A6a prefilter: the first few points decide most rotations (off the road)
        for (int k = tid; k <= K; k += nt) s_flags[k] = 0;
        OdMap m;
        {
            const int msel = cc.map_sel;
            const int* dims = e.od_map_dims + ((size_t)b * 2 + msel) * 4;
            m.sx = dims[0]; m.sy = dims[1]; m.mx = (double)dims[2]; m.my = (double)dims[3];
            m.map = e.od_maps + e.od_map_off[(size_t)b * 2 + msel];
        }
        __syncthreads();
        const int npre = min(ob.count, ONMAP_PRE_PTS);
        for (int k = 1 + tid; k <= K; k += nt) {
            bool any_in = false, bad = false;
            thread_onmap_od(m, ox, oy, 0, npre, e.cos_k[k], e.sin_k[k], any_in, bad);
            if (!bad) s_flags[k] = CF_PRE;
        }
        __syncthreads();
        n_list = block_compact(s_flags, K, CF_PRE, CF_PRE, s_list, c.s_warp);
        if (tid == 0) atomicAdd(&e.stats[6], (unsigned long long)n_list);
    } else {
        __syncthreads();
    }
    clk.lap(e, WT_SETUP);
    const int g = tid / GRP, gl = tid % GRP;
    const unsigned gm = group_mask();
    const int min_pts = max(cc.min_points, 1);                     // od/ins:530: V == 0 or V < min_points -> rejected
    const ImageGeom geom = s.geom;
    const FastGeom fgeom = make_fast_geom(geom);
    const double* smooth = e.smooth + (size_t)b * e.hw;
    // Stage A (the map test of a window of candidates) feeds a queue of on-map candidates in yaw order; stages B + C take
    // them off the queue in CHUNKS of one candidate per warp: road level (OD) -> collision test -> occlusion count of the
    // chunk's feasible candidates, leaving at the first candidate that keeps min_points (od/ins:530-561).  The first
    // feasible candidates of a try are the likely winners, so the first chunk runs on whatever the first non-empty window
    // yields; after that (OD) stage A runs ahead until a whole chunk is waiting, so that a sparse window does not cost a
    // round of road levels / collisions / occlusion for two candidates.  Semseg keeps window-by-window chunks: its stage
    // A already carries the road levels (the z shift walks from yaw to yaw).
    int base = 0, q_head = 0, q_n = 0, ss_c0 = 0, ss_n = 0;
    bool first_chunk = true;
    for (;;) {
        const int* chunk;
        int nch;
        if (e.task == 0) {
            while (base < n_list && (first_chunk ? q_n == 0 : q_n < WALK_NWARPS)) {
                const int nw = min(WALK_W, n_list - base);
                if (g < nw) {                                 // A5 + A6a on every object point, an 8-lane group per candidate
                    const int k = s_list[base + g];
                    const bool on = walk_onmap_od(e, b, ob, cc, ox, oy, k, gl, gm);
                    if (gl == 0) {
                        const double ck = e.cos_k[k], sk = e.sin_k[k];
                        c.a_k[g] = k; c.a_on[g] = on ? 1 : 0;
                        c.a_cx[g] = sub(mul(ck, ob.cx), mul(sk, ob.cy)); c.a_cy[g] = add(mul(sk, ob.cx), mul(ck, ob.cy));
                    }
                }
                __syncthreads();
                if (tid == 0) { const long long n = clock64(); atomicAdd(&e.stats[WALK_T0 + WT_ONMAP], (unsigned long long)(n - clk.t)); }
                const int n_on = walk_window_list(c, nw, c.won, [&](int i) { return c.a_on[i] != 0; });
                if (tid < n_on) {                             // append to the queue (a ring over the candidate records)
                    const int slot = (q_head + q_n + tid) % WALK_Q, i = c.won[tid];
                    c.wk[slot] = c.a_k[i]; c.wflag[slot] = CF_ONMAP; c.wlevel[slot] = 0.0; c.wcx[slot] = c.a_cx[i]; c.wcy[slot] = c.a_cy[i];
                }
                if (tid == 0) { atomicAdd(&e.stats[7], (unsigned long long)n_on); atomicAdd(&e.stats[9], 1ull); }
                __syncthreads();
                q_n += n_on;
                base += WALK_W;
            }
            if (q_n == 0) break;
            nch = min(WALK_NWARPS, q_n);
            if (tid < nch) c.wlist[tid] = (q_head + tid) % WALK_Q;
            if (tid == 0) c.next = 0;
            __syncthreads();
            chunk = c.wlist;
        } else {
            while (ss_c0 >= ss_n && base < n_list) {
                ss_n = walk_window_ss(e, b, s, c, ox, oy, oz, base, min(WALK_W, n_list - base));
                ss_c0 = 0;
                base += WALK_W;
                if (tid == 0) atomicAdd(&e.stats[9], 1ull);
            }
            if (ss_c0 >= ss_n) break;
            nch = min(WALK_NWARPS, ss_n - ss_c0);
            chunk = c.won + ss_c0;
        }
        {
            if (e.task == 0) {
                walk_levels(e, b, c, chunk, nch);
                __syncthreads();
            }
            if (tid == 0) {                                   // the chunk's candidates with a road level, in order
                int n = 0;
                for (int t = 0; t < nch; ++t)
                    if ((c.wflag[chunk[t]] & (CF_ONMAP | CF_HOK)) == (CF_ONMAP | CF_HOK)) { c.whit[chunk[t]] = 0; c.wsub[n++] = chunk[t]; }
                c.n_sub = n; c.next = 0;
            }
            __syncthreads();
            walk_collides(e, b, s, c, c.wsub, c.n_sub);
            __syncthreads();
            clk.lap(e, WT_PLACE);
            if (tid == 0) {                                   // feasible candidates of the chunk in rotation order (od/fs:288-296)
                int n = 0;
                for (int t = 0; t < c.n_sub; ++t)
                    if ((c.wflag[c.wsub[t]] & (CF_ONMAP | CF_HOK | CF_COLLIDE)) == (CF_ONMAP | CF_HOK)) c.wfeas[n++] = c.wsub[t];
                c.nfw = n; c.next = 0;
                if (n) { c.last_k = c.wk[c.wfeas[n - 1]]; c.last_level = c.wlevel[c.wfeas[n - 1]]; }
                c.n_feas += n;
            }
            __syncthreads();
            // stage C: A11 in rotation order with an early exit.  lo = points that are individually closer than the
            // scene, hi = points that fall into the image: lo <= V <= hi, and lo == 0 <=> V == 0, so most candidates are
            // decided without building the visible-pixel image
            const int nfw = c.nfw;
            for (int j0 = 0, npar = 1; j0 < nfw && c.found < 0; j0 += npar) {
                // candidates counted side by side: as many as are left (at most WALK_OCC_PAR), rounded up to a divisor of
                // the warp count so that every candidate gets whole warps — a lone feasible candidate gets the whole CTA
                npar = 1;
                while (npar < min(nfw - j0, WALK_OCC_PAR) || WALK_NWARPS % npar != 0) ++npar;
                const int lanes = WALK_THREADS / npar, sg = tid / lanes, sl = tid % lanes;
                if (tid < WALK_OCC_PAR) { c.cnt_lo[tid] = 0; c.cnt_hi[tid] = 0; }
                __syncthreads();
                const int j = j0 + sg;
                if (j < nfw) {
                    const int i = c.wfeas[j], k = c.wk[i];
                    const double cs = e.cos_k[k], sn = e.sin_k[k], dz = sub(c.wlevel[i], ob.cz);
                    int lo = 0, hi = 0;
                    for (int p = sl; p < ob.count; p += lanes) {
                        const ObjPix o = project_obj_pix(e, ob, geom, fgeom, p, cs, sn, dz, s);
                        if (o.pix >= 0) { ++hi; if (o.r < smooth[o.pix]) ++lo; }
                    }
                    for (int o = 16; o > 0; o >>= 1) { lo += __shfl_xor_sync(0xffffffffu, lo, o); hi += __shfl_xor_sync(0xffffffffu, hi, o); }
                    if ((tid & 31) == 0) { if (lo) atomicAdd(&c.cnt_lo[sg], lo); if (hi) atomicAdd(&c.cnt_hi[sg], hi); }
                }
                __syncthreads();
                int found = -1;
                for (int q = 0; q < npar && j0 + q < nfw; ++q) {                  // uniform over the CTA
                    const int lo = c.cnt_lo[q], hi = c.cnt_hi[q];
                    bool ok = lo >= min_pts;
                    if (!ok && lo > 0 && hi >= min_pts) {
                        const int i = c.wfeas[j0 + q];
                        ok = walk_exact_visible(e, b, s, c, c.wk[i], c.wlevel[i], reinterpret_cast<unsigned*>(scratch)) >= min_pts;
                    }
                    if (ok) { found = j0 + q; break; }
                }
                if (found >= 0 && tid == 0) {
                    const int i = c.wfeas[found];
                    c.found = found; c.found_k = c.wk[i]; c.found_level = c.wlevel[i];
                }
                __syncthreads();
            }
            clk.lap(e, WT_OCCL);
        }
        if (c.found >= 0) break;
        if (e.task == 0) { q_head = (q_head + nch) % WALK_Q; q_n -= nch; first_chunk = false; }
        else ss_c0 += nch;
    }
    // A11 + A12 for the chosen candidate: the first one that keeps min_points, else the last feasible one (its
    // vis_px still deletes scene points in the reference, od/ins:472-501)
    const int n_feas = c.n_feas;
    if (tid == 0) s.n_feasible = n_feas;
    if (n_feas > 0) {
        const bool accepted = c.found >= 0;
        const int k = accepted ? c.found_k : c.last_k;
        if (tid == 0) e.cand_level[(size_t)b * (K + 1) + k] = accepted ? c.found_level : c.last_level;
        __syncthreads();
        select_emit_body(e, b, s, k, accepted,
                         sel_scratch(reinterpret_cast<unsigned long long*>(dyn), WALK_SEL_KEYS, WALK_SEL_PTS, WALK_SEL_TILE));
    }
    __syncthreads();
    if (e.task == 1 && n_feas > 0 && c.found >= 0) {               // the appended object points join the map marks (next slot)
        const double* T = e.poses + (size_t)b * 16;
        for (int p = s.n0 + s.tail_before + tid; p < s.n0 + s.n_tail; p += nt) adjust_map_point(e, b, s, T, p, 1, true);
        __syncthreads();
    }
    clk.lap(e, WT_SELECT);
}

__global__ void __launch_bounds__(WALK_THREADS, WALK_CTAS_PER_SM) k_scan_walk(const __grid_constant__ EngineDev e, int n_scans) {
    const int b = blockIdx.x;
    if (b >= n_scans) return;
    extern __shared__ __align__(16) unsigned char w_dyn[];
    __shared__ WalkCtl c;
    // the scan's scheduling state lives in shared memory while its CTA runs: the serial scheduling step and every stage
    // read and write it dozens of times
    __shared__ ScanState s;
    {
        const int* src = reinterpret_cast<const int*>(&e.st[b]);
        int* dst = reinterpret_cast<int*>(&s);
        for (int i = threadIdx.x; i < (int)(sizeof(ScanState) / sizeof(int)); i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x == 0) s.far_flag = e.task == 1 && e.occ_far[(size_t)b * (OCC_FAR_CAP + 1)] != 0;
    __syncthreads();
    const WalkSmem L = walk_smem_layout(e.K, e.dwords);
    int steps = 0;
    WalkClock clk;
    clk.start();
    const long long t_begin = clk.t;
    for (;;) {
        if (threadIdx.x == 0) {
            int apply = 0, project = 0, tryact = 0;
            ctrl_advance(e, b, s, apply, project, tryact);
            c.apply = apply; c.project = project; c.tryact = tryact;
            if (apply) atomicAdd(&e.stats[2], 1ull);
        }
        __syncthreads();
        const int apply = c.apply, project = c.project, tryact = c.tryact;
        clk.lap(e, WT_CTRL);
        if (apply || project) walk_update(e, b, s, c, apply, project, w_dyn + L.scratch_off, w_dyn);
        clk.lap(e, WT_UPDATE);
        if (!tryact) break;                              // PH_DONE or PH_ERROR
        walk_try(e, b, s, c, w_dyn, L, clk);
        ++steps;
    }
    if (threadIdx.x == 0) {
        const long long lived = clock64() - t_begin;
        atomicAdd(&e.stats[WALK_T0 + WT_TOTAL], (unsigned long long)lived);
        s.walk_cycles = lived; s.walk_tries = steps;
    }
    __syncthreads();
    {
        const int* src = reinterpret_cast<const int*>(&s);
        int* dst = reinterpret_cast<int*>(&e.st[b]);
        for (int i = threadIdx.x; i < (int)(sizeof(ScanState) / sizeof(int)); i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x == 0) atomicMax(&e.stats[8], (unsigned long long)steps);
}

// what the first round of the staged engine sets up, for the walker: every scan is listed for the batch-wide full
// projection and every tile for close/fill; the state machine starts with its first range image already built
__global__ void k_walk_prepare(EngineDev e, int n_scans, int reset_range) {
    const int tiles = e.cf_tiles;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_scans * tiles; i += gridDim.x * blockDim.x) e.cf_tasks[i] = i;
    for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < n_scans; b += gridDim.x * blockDim.x) {
        e.full_list[b] = b;
        e.gate_update[b] = 1;                            // k_adjust_map (semseg) runs for every scan
        if (e.task == 1) for (int i = 0; i <= OCC_FAR_CAP; ++i) occ_far_clear(e, b, i);
        ScanState& s = e.st[b];
        s.first = 0; s.scene_changed = 0;
        if (reset_range) { s.min_el_bits = R3D_EMPTY_U64; s.max_el_bits = 0ull; }      // k_minmax follows
        atomicAdd(&e.stats[0], 1ull);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) { e.work_cnt[0] = n_scans; e.work_cnt[1] = n_scans * tiles; e.stats[8] = 0ull; }
}
