// Kernels of the batched Real3D-Aug engine, part: the fused once-per-scan streaming passes.
// Included by r3d_engine_kernels.cuh (inside namespace r3d, after r3d_k_grid.cuh); not a standalone header.
// ------------------------------------------------------------------------------------------------ prepass
// Two passes over the float4 points instead of the seven of the first version (ingest, grid count, index count, grid
// scatter, index scatter, min/max, projection):
//   k_ingest_count     A1 + A2 (r, elevation, azimuth bin cached), min / max elevation of the scan, per-cell /
//                      per-column-group COUNTS of the three CSR indices, z-buffer cleared on the side
//   k_bucket_scan3     exclusive scans of the three count arrays (one launch)
//   k_scatter_project  CSR scatter of the three indices + A3 (pix ids, 64-bit atomicMin z-buffer)
// Consecutive points of a spinning LiDAR fall into the same 0.5 m cell / column group, so the histogram atomics are
// aggregated per warp with __match_any_sync: one atomic per distinct key of the warp instead of one per point.
// Timing-only ablations for tools/gpu_prepass_ab.sh (variant builds only, their outputs are wrong): R3D_ABLATE_COL_IDX
// drops the col_idx store, R3D_ABLATE_COL_ATOMICS the column count / slot atomics (and with them the col_idx store),
// R3D_ABLATE_GRID_STORES the two grid-entry stores.
__device__ __forceinline__ void agg_count(int* arr, int key, bool active) {
    const unsigned act = __ballot_sync(0xffffffffu, active);
    if (!active) return;
    const unsigned peers = __match_any_sync(act, key);
    if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&arr[key], __popc(peers));
}
__device__ __forceinline__ int agg_slot(int* arr, int key, bool active) {
    const unsigned act = __ballot_sync(0xffffffffu, active);
    if (!active) return -1;
    const unsigned peers = __match_any_sync(act, key);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(&arr[key], __popc(peers));
    base = __shfl_sync(peers, base, leader);
    return base + __popc(peers & ((1u << lane) - 1u));
}

// the same in two halves: the returning atomic of the group's leader is issued at once, its result is only waited for
// when the slot is needed — so the round trips of several indices / points overlap
struct AggTicket { unsigned peers; int base; };
__device__ __forceinline__ AggTicket agg_issue(int* arr, int key, bool active) {
    AggTicket t{0u, 0};
    const unsigned act = __ballot_sync(0xffffffffu, active);
    if (active) {
        t.peers = __match_any_sync(act, key);
        if ((int)(threadIdx.x & 31) == __ffs(t.peers) - 1) t.base = atomicAdd(&arr[key], __popc(t.peers));
    }
    return t;
}
__device__ __forceinline__ int agg_finish(const AggTicket& t) {
    if (!t.peers) return -1;
    const int base = __shfl_sync(t.peers, t.base, __ffs(t.peers) - 1);
    return base + __popc(t.peers & ((1u << (threadIdx.x & 31)) - 1u));
}

// OD: a point goes to the all-points grid (not Road) or to the surface grid (Road, z > -3), never to both, so ONE
// aggregated atomic serves the two grids: which = 0 (all-points), 1 (surface), -1 (neither)
__device__ __forceinline__ bool grids_exclusive(const EngineDev& e) {
    return e.task == 0 && e.n_surf_all == 1 && e.surf_all[0] == e.road_label;
}
__device__ __forceinline__ void agg_count2(int* arr_a, int* arr_g, int gc, int which) {
    const unsigned act = __ballot_sync(0xffffffffu, which >= 0);
    if (which < 0) return;
    const unsigned peers = __match_any_sync(act, gc * 2 + which);
    if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&(which ? arr_g : arr_a)[gc], __popc(peers));
}
__device__ __forceinline__ AggTicket agg_issue2(int* arr_a, int* arr_g, int gc, int which) {
    AggTicket t{0u, 0};
    const unsigned act = __ballot_sync(0xffffffffu, which >= 0);
    if (which >= 0) {
        t.peers = __match_any_sync(act, gc * 2 + which);
        if ((int)(threadIdx.x & 31) == __ffs(t.peers) - 1) t.base = atomicAdd(&(which ? arr_g : arr_a)[gc], __popc(t.peers));
    }
    return t;
}

__global__ void __launch_bounds__(STREAM_THREADS) k_ingest_count(EngineDev e, int n_scans) {
    const int b = blockIdx.y;
    if (b >= n_scans) return;
    ScanState& s = e.st[b];
    const int n0 = s.n0;
    const int p0 = blockIdx.x * CHUNK;
    {   // this CTA's share of the scan's z-buffer (od/ins:99: train = 500 everywhere = "empty")
        unsigned long long* z = e.zraw + (size_t)b * e.hw;
        const int per = (e.hw + gridDim.x - 1) / gridDim.x;
        for (int i = blockIdx.x * per + threadIdx.x; i < min((int)(blockIdx.x + 1) * per, e.hw); i += STREAM_THREADS) z[i] = R3D_EMPTY_U64;
    }
    if (p0 >= n0) return;
    const double d_az = kTwoPi / (double)e.cols;
    const float inv_d_az = (float)(1.0 / d_az);
    float err_az = 6e-6f * inv_d_az + 5e-7f * (float)e.cols + 1e-5f;       // r3d_common.cuh, fast binning
    if (!(err_az < 0.25f)) err_az = 2.0f;
    const size_t base = (size_t)b * e.P;
    int* cell = e.gcell + (size_t)b * e.G * e.G;
    int* acell = e.acell + (size_t)b * e.G * e.G;
    int* coff = e.col_off + (size_t)b * (col_groups(e.cols) + 1);
    unsigned long long lmin = R3D_EMPTY_U64, lmax = 0ull;
    const bool excl = grids_exclusive(e);
    const float4* __restrict__ src = e.xyzi + (size_t)b * e.max_points;
    const int q_end = min(p0 + CHUNK, n0);
    // the next point's loads are issued before the arithmetic of the current one (~500 instructions) starts
    float4 vn = make_float4(1.f, 0.f, 0.f, 0.f);
    unsigned labn = 0u;
    if (p0 + (int)threadIdx.x < n0) { vn = __ldg(&src[p0 + threadIdx.x]); labn = e.label[base + p0 + threadIdx.x]; }
    for (int q = p0; q < q_end; q += STREAM_THREADS) {       // whole warps stay in the loop (aggregated atomics)
        const int p = q + threadIdx.x;
        const bool in = p < n0;
        const float4 v = vn;
        const unsigned lab = labn;
        {
            const int pn = p + STREAM_THREADS;
            vn = make_float4(1.f, 0.f, 0.f, 0.f); labn = 0u;
            if (q + STREAM_THREADS < q_end && pn < n0) { vn = __ldg(&src[pn]); labn = e.label[base + pn]; }
        }
        const double x = v.x, y = v.y, z = v.z;
        const double r = range3(x, y, z);
        const double el = elevation(z, r);
        int c;
        if (!fast_col(inv_d_az, err_az, e.cols, v.x, v.y, c)) c = trunc_to_int(__ddiv_rn(az_mod(azimuth(x, y)), d_az));
        const int cc = max(0, min(c, e.cols - 1));
        if (in) {
            if (!(r > 0.0) || c < 0 || c >= e.cols) set_error(s, R3D_ERR_ASSERT);      // od/ins:113 / nan elevation
            e.r[base + p] = r;
            e.el[base + p] = el;
            e.col[base + p] = (unsigned short)cc;
            e.alive[base + p] = 1;
            const unsigned long long bits = dbl_bits(el);
            lmin = min(lmin, bits); lmax = max(lmax, bits);
        }
        const int gc = grid_coord(e, v.y) * e.G + grid_coord(e, v.x);
        const bool in_a = in && !(e.task == 0 && lab == (unsigned)e.road_label);         // od/ins:353-355
        const bool in_g = in && (double)v.z > -3.0 && any_surface_label(e, lab);         // od/fs:154-155
        if (excl) agg_count2(acell, cell, gc, in_g ? 1 : (in_a ? 0 : -1));
        else { agg_count(acell, gc, in_a); agg_count(cell, gc, in_g); }
#ifndef R3D_ABLATE_COL_ATOMICS
        agg_count(coff, cc / COL_GROUP, in);
#endif
    }
    __shared__ unsigned long long s_min[STREAM_THREADS / 32], s_max[STREAM_THREADS / 32];
    for (int o = 16; o > 0; o >>= 1) {
        lmin = min(lmin, __shfl_xor_sync(0xffffffffu, lmin, o));
        lmax = max(lmax, __shfl_xor_sync(0xffffffffu, lmax, o));
    }
    if ((threadIdx.x & 31) == 0) { s_min[threadIdx.x >> 5] = lmin; s_max[threadIdx.x >> 5] = lmax; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < STREAM_THREADS / 32; ++w) { lmin = min(lmin, s_min[w]); lmax = max(lmax, s_max[w]); }
        // A2 (od/ins:79-80): every original point is live at this time (k_reset_state armed the two words)
        if (lmax >= lmin) { atomicMin(&s.min_el_bits, lmin); atomicMax(&s.max_el_bits, lmax); }
    }
}

// the three exclusive scans (surface grid, all-points grid, column groups) in one launch: blockIdx.y selects the array
__global__ void __launch_bounds__(1024) k_bucket_scan3(EngineDev e, int n_scans) {
    const size_t gg = (size_t)e.G * e.G;
    if (blockIdx.y == 0) bucket_scan_body(e.gcell, gg, (int)gg, n_scans);
    else if (blockIdx.y == 1) bucket_scan_body(e.acell, gg, (int)gg, n_scans);
    else bucket_scan_body(e.col_off, (size_t)col_groups(e.cols) + 1, col_groups(e.cols), n_scans);
}

__global__ void __launch_bounds__(STREAM_THREADS) k_scatter_project(EngineDev e, int n_scans) {
    const int b = blockIdx.y;
    if (b >= n_scans) return;
    ScanState& s = e.st[b];
    const int n0 = s.n0;
    const int p0 = blockIdx.x * CHUNK;
    if (blockIdx.x == 0 && threadIdx.x == 0) {           // what k_clear_images does for a full projection
        e.far_arr[b] = 0;
        if (s.min_el_bits == R3D_EMPTY_U64) set_error(s, R3D_ERR_ASSERT);
        s.geom = make_geom(e.rows, e.cols, e.cols, bits_dbl(s.max_el_bits), bits_dbl(s.min_el_bits));
    }
    if (p0 >= n0) return;
    const ImageGeom g = make_geom(e.rows, e.cols, e.cols, bits_dbl(s.max_el_bits), bits_dbl(s.min_el_bits));
    const size_t base = (size_t)b * e.P;
    int* cell = e.gcell + (size_t)b * e.G * e.G;
    int* acell = e.acell + (size_t)b * e.G * e.G;
    int* coff = e.col_off + (size_t)b * (col_groups(e.cols) + 1);
    float4* out = e.gpts + (size_t)b * e.max_points;
    float4* aout = e.apts + (size_t)b * e.max_points;
    int* cidx = e.col_idx + (size_t)b * e.max_points;
    unsigned long long* z = e.zraw + (size_t)b * e.hw;
    static_assert(CHUNK % (2 * STREAM_THREADS) == 0, "two points per thread and iteration");
    const bool excl = grids_exclusive(e);
    for (int q = p0; q < min(p0 + CHUNK, n0); q += 2 * STREAM_THREADS) {
        // two points per thread: all loads first, then the six slot atomics back to back, then the stores
        int p[2], col[2], gc[2], which[2];
        bool in[2];
        float4 v[2];
        unsigned lab[2];
        double el[2], r[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            p[u] = q + u * STREAM_THREADS + threadIdx.x;
            in[u] = p[u] < n0;
            v[u] = make_float4(1.f, 0.f, 0.f, 0.f); lab[u] = 0u; col[u] = 0; el[u] = 0.0; r[u] = 0.0;
            if (in[u]) {
                v[u] = __ldg(&e.xyzi[(size_t)b * e.max_points + p[u]]); lab[u] = e.label[base + p[u]]; col[u] = e.col[base + p[u]];
                el[u] = e.el[base + p[u]]; r[u] = e.r[base + p[u]];
            }
        }
        AggTicket ta[2], tg[2], tc[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            gc[u] = grid_coord(e, v[u].y) * e.G + grid_coord(e, v[u].x);
            const bool in_a = in[u] && !(e.task == 0 && lab[u] == (unsigned)e.road_label);
            const bool in_g = in[u] && (double)v[u].z > -3.0 && any_surface_label(e, lab[u]);
            if (excl) {                                  // one atomic for the two grids (see agg_count2)
                which[u] = in_g ? 1 : (in_a ? 0 : -1);
                ta[u] = agg_issue2(acell, cell, gc[u], which[u]);
                tg[u] = AggTicket{0u, 0};
            } else {
                which[u] = -1;
                ta[u] = agg_issue(acell, gc[u], in_a);
                tg[u] = agg_issue(cell, gc[u], in_g);
            }
#ifndef R3D_ABLATE_COL_ATOMICS
            tc[u] = agg_issue(coff, col[u] / COL_GROUP, in[u]);
#else
            tc[u] = AggTicket{0u, 0};
#endif
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            int pix = -1;
            if (in[u]) {                                 // A3 (od/ins:85-130)
                const int row = bin_row(g, el[u]);
                if (row < 0 || row >= g.rows) set_error(s, R3D_ERR_ASSERT);             // od/ins:111
                else { pix = row * g.cols + col[u]; atomicMin(&z[pix], dbl_bits(r[u])); }
                e.pix[base + p[u]] = pix;
            }
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int sa = agg_finish(ta[u]), sg = agg_finish(tg[u]);
#ifndef R3D_ABLATE_GRID_STORES
            if (sa >= 0) {
                if (which[u] == 1) out[sa] = make_float4(v[u].x, v[u].y, v[u].z, __uint_as_float(lab[u]));
                else aout[sa] = make_float4(v[u].x, v[u].y, v[u].z, apt_tag(e, lab[u], p[u]));
            }
            if (sg >= 0) out[sg] = make_float4(v[u].x, v[u].y, v[u].z, __uint_as_float(lab[u]));
#else
            if (sa + sg == -3) cidx[0] = p[u];          // never true: keeps the grid slot atomics returning ones
#endif
            const int sc = agg_finish(tc[u]);
#ifndef R3D_ABLATE_COL_IDX
            if (sc >= 0) cidx[sc] = p[u];
#else
            if (sc == -2) cidx[0] = p[u];                // never true: keeps the slot atomic a returning one
#endif
        }
    }
}

// Chebyshev distance (in cells, capped at NEAR_CAP) from every cell of the surface grid to the nearest non-empty one.
// One CTA per scan, bit-parallel: the occupancy of the grid is a bit image in shared memory (a row of G cells = a few
// 32-bit words); dilating it by a 3 x 3 square d times gives the cells within Chebyshev distance d, so the distance of a
// cell is the first d at which its bit turns on — a dozen sweeps of shifts and ORs over ~2k words instead of a 23-tap
// min filter per cell in each direction.
constexpr int NEAR_THREADS = 1024;
__host__ __device__ __forceinline__ size_t grid_near_smem(int G) {
    const int wpr = (G + 31) / 32;
    return (size_t)G * G + 2 * (size_t)(G + 2) * wpr * 4;           // distance bytes + two bit images with a zero row above / below
}
__global__ void __launch_bounds__(NEAR_THREADS) k_grid_near_bits(EngineDev e, int n_scans) {
    const int b = blockIdx.x, G = e.G;
    if (b >= n_scans) return;
    extern __shared__ __align__(16) unsigned char s_near[];
    const int wpr = (G + 31) / 32, nwords = G * wpr;
    unsigned char* s_dist = s_near;                                              // [G][G]
    unsigned* s_a = reinterpret_cast<unsigned*>(s_near + (((size_t)G * G + 15) & ~(size_t)15));   // [(G + 2)][wpr], row 0 and G + 1 stay zero
    unsigned* s_b = s_a + (size_t)(G + 2) * wpr;
    const int* cell = e.gcell + (size_t)b * G * G;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = NEAR_THREADS / 32;
    for (int i = tid; i < (G + 2) * wpr; i += NEAR_THREADS) { s_a[i] = 0u; s_b[i] = 0u; }
    for (int i = tid; i < G * G / 4; i += NEAR_THREADS) reinterpret_cast<unsigned*>(s_dist)[i] = 0x01010101u * (unsigned)NEAR_CAP;
    for (int i = (G * G / 4) * 4 + tid; i < G * G; i += NEAR_THREADS) s_dist[i] = (unsigned char)NEAR_CAP;
    __syncthreads();
    for (int u = warp; u < nwords; u += nwarps) {                                // occupancy bits, one ballot per word
        const int y = u / wpr, x = (u % wpr) * 32 + lane;
        bool occ = false;
        if (x < G) { const int q = y * G + x; occ = cell[q] > (q > 0 ? cell[q - 1] : 0); }
        const unsigned m = __ballot_sync(0xffffffffu, occ);
        if (lane == 0) s_a[(size_t)(y + 1) * wpr + u % wpr] = m;
        if (occ) s_dist[y * G + x] = 0;
    }
    __syncthreads();
    unsigned* cur = s_a;
    unsigned* nxt = s_b;
    for (int d = 1; d < NEAR_CAP; ++d) {
        for (int u = tid; u < nwords; u += NEAR_THREADS) {
            const int y = u / wpr, w = u % wpr;
            unsigned acc = 0u;
#pragma unroll
            for (int dy = 0; dy <= 2; ++dy) {                                    // rows y - 1, y, y + 1 (padded image)
                const unsigned* row = cur + (size_t)(y + dy) * wpr;
                const unsigned m = row[w];
                acc |= m | (m << 1) | (m >> 1) | (w > 0 ? row[w - 1] >> 31 : 0u) | (w + 1 < wpr ? row[w + 1] << 31 : 0u);
            }
            if (w == wpr - 1 && (G & 31)) acc &= (1u << (G & 31)) - 1u;            // no cells beyond column G - 1
            const unsigned old = cur[(size_t)(y + 1) * wpr + w];
            nxt[(size_t)(y + 1) * wpr + w] = acc;
            unsigned fresh = acc & ~old;                                          // cells first reached at distance d
            while (fresh) {
                const int bit = __ffs(fresh) - 1; fresh &= fresh - 1;
                const int x = w * 32 + bit;
                if (x < G) s_dist[y * G + x] = (unsigned char)d;
            }
        }
        __syncthreads();
        unsigned* t = cur; cur = nxt; nxt = t;
    }
    unsigned char* out = e.gnear + (size_t)b * G * G;
    if ((((size_t)b * G * G) & 15) == 0 && (G * G) % 16 == 0) {
        for (int i = tid; i < G * G / 16; i += NEAR_THREADS) reinterpret_cast<uint4*>(out)[i] = reinterpret_cast<const uint4*>(s_dist)[i];
    } else {
        for (int i = tid; i < G * G; i += NEAR_THREADS) out[i] = s_dist[i];
    }
}
