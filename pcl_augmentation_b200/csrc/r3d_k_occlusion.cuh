// Kernels of the batched Real3D-Aug engine, part: A10 - A12 occlusion count, candidate selection, insertion.
// Included by r3d_engine_kernels.cuh (inside namespace r3d, after the shared constants); not a standalone header.
// ------------------------------------------------------------------------------------------- occlusion
// object point i of candidate k -> (pix, r) in the CURRENT scene geometry (od/ins:474-478, sample=True)
struct ObjProj { double x, y, z, r, el; int pix, col; };
__device__ __forceinline__ ObjProj project_obj_point(const EngineDev& e, const ObjBox& ob, const ImageGeom& g, int i,
                                                     double c, double sn, double dz, ScanState& s) {
    ObjProj o;
    const double x0 = e.obj_x[ob.first + i], y0 = e.obj_y[ob.first + i];
    o.x = sub(mul(c, x0), mul(sn, y0));
    o.y = add(mul(sn, x0), mul(c, y0));
    o.z = add(e.obj_z[ob.first + i], dz);
    o.r = range3(o.x, o.y, o.z);
    o.el = elevation(o.z, o.r);
    const int row = bin_row(g, o.el);
    o.col = bin_col(g, azimuth(o.x, o.y));
    o.pix = -1;
    if (row >= 0 && row < g.rows) {                                    // od/ins:108-109
        if (o.col < 0 || o.col >= g.cols) set_error(s, R3D_ERR_ASSERT);  // od/ins:113
        else o.pix = row * g.cols + o.col;
    }
    return o;
}

// the same for the occlusion counts, which need the pixel and the range only: the bins come from the float estimate of
// the angles where that is safe (r3d_common.cuh, fast binning), else from the exact path above
struct ObjPix { double r; int pix; };
__device__ __forceinline__ ObjPix project_obj_pix(const EngineDev& e, const ObjBox& ob, const ImageGeom& g, const FastGeom& fg, int i,
                                                  double c, double sn, double dz, ScanState& s) {
    ObjPix o;
    const double x0 = e.obj_x[ob.first + i], y0 = e.obj_y[ob.first + i];
    const double x = sub(mul(c, x0), mul(sn, y0)), y = add(mul(sn, x0), mul(c, y0)), z = add(e.obj_z[ob.first + i], dz);
    o.r = range3(x, y, z);
    int row, col;
    if (!fast_row(fg, g.rows, (float)z, (float)o.r, row)) row = bin_row(g, elevation(z, o.r));
    if (!fast_col(fg.inv_d_az, fg.err_az, g.cols, (float)x, (float)y, col)) col = bin_col(g, azimuth(x, y));
    o.pix = -1;
    if (row >= 0 && row < g.rows) {                                    // od/ins:108-109
        if (col < 0 || col >= g.cols) set_error(s, R3D_ERR_ASSERT);      // od/ins:113
        else o.pix = row * g.cols + col;
    }
    return o;
}

// A11 (od/ins:486-501) for every feasible candidate: V = number of object points whose pixel is visible.  A pixel
// that holds object points keeps its own min range through smooth_out, and min_r < scene <=> some point of the pixel
// has r < scene, so no z-buffer is needed for the count: pass 1 marks visible pixels in a shared-memory bit image,
// pass 2 counts the points on marked pixels.  Candidates are visited in rotation order with an ordered early-out
// (the reference stops at the first candidate that keeps >= min_points, od/ins:530-561).
__global__ void k_phase_gate(EngineDev e, int n_scans) {           // which scans found nothing in the first window
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b < n_scans) e.need2[b] = e.gate_try[b] && e.st[b].found_rank == INT_MAX && e.n_list[b] > e.cand_window;
}

__global__ void __launch_bounds__(128) k_occl_count(EngineDev e, int n_scans, int phase) {
    const int b = blockIdx.y;
    if (b >= n_scans || !(phase == 2 ? e.need2[b] : e.gate_try[b])) return;
    ScanState& s = e.st[b];
    extern __shared__ unsigned s_bits[];
    __shared__ int s_cnt, s_stop;
    __shared__ int s_warp[4];
    // ordered list of the feasible rotations (the order find_possible_places returns them, od/fs:288-296): every CTA
    // of the scan compacts the flag bytes itself; the first one publishes the list for k_select_emit
    unsigned short* s_feas = reinterpret_cast<unsigned short*>(s_bits + e.dwords);
    const size_t cb = (size_t)b * (e.K + 1);
    const int nf = block_compact(e.cand_flags + cb, e.K, CF_ONMAP | CF_HOK | CF_COLLIDE, CF_ONMAP | CF_HOK, s_feas, s_warp);
    if (blockIdx.x == 0) {
        for (int i = threadIdx.x; i < nf; i += blockDim.x) e.feas[(size_t)b * e.K + i] = s_feas[i];
        if (threadIdx.x == 0) s.n_feasible = nf;
    }
    if ((int)blockIdx.x >= nf) return;
    for (int i = threadIdx.x; i < e.dwords; i += blockDim.x) s_bits[i] = 0u;
    const ObjBox ob = e.try_obj[b];
    const int min_pts = e.classes[ob.cls].min_points;
    const ImageGeom g = s.geom;
    const double* smooth = e.smooth + (size_t)b * e.hw;
    int* pixbuf = e.occ_pix + ((size_t)b * OCC_G + blockIdx.x) * e.max_obj_points;
    __syncthreads();
    for (int rank = blockIdx.x; rank < nf; rank += gridDim.x) {
        if (threadIdx.x == 0) { s_stop = *(volatile int*)&s.found_rank < rank; s_cnt = 0; }
        __syncthreads();
        if (s_stop) break;                                        // an earlier candidate already passed
        const int k = s_feas[rank];
        const double c = e.cos_k[k], sn = e.sin_k[k];
        const double dz = sub(e.cand_level[cb + k], ob.cz);
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const ObjProj o = project_obj_point(e, ob, g, i, c, sn, dz, s);
            pixbuf[i] = o.pix;
            if (o.pix >= 0 && o.r < smooth[o.pix]) atomicOr(&s_bits[o.pix >> 5], 1u << (o.pix & 31));
        }
        __syncthreads();
        int cnt = 0;
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const int pix = pixbuf[i];
            if (pix >= 0 && (s_bits[pix >> 5] & (1u << (pix & 31)))) ++cnt;
        }
        for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        if ((threadIdx.x & 31) == 0 && cnt) atomicAdd(&s_cnt, cnt);
        __syncthreads();
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const int pix = pixbuf[i];
            if (pix >= 0) s_bits[pix >> 5] = 0u;
        }
        if (threadIdx.x == 0) {
            e.cand_v[cb + k] = s_cnt;
            if (s_cnt > 0 && s_cnt >= min_pts) atomicMin(&s.found_rank, rank);      // od/ins:530-536
        }
        __syncthreads();
    }
}

// smoothed object range at pixel (r, c): own min range, or the neighbour mean where the 5x3 closing switches an
// empty pixel on (cl:26-62).  `dil` is the bit image of the dilated occupancy (union of the 5x3 neighbourhoods of the
// object's pixels), so closed(q) = AND of dil over the in-image 5x3 neighbourhood of q.
__device__ bool obj_pixel_value(const unsigned long long* raw, const unsigned* dil, int H, int W, int r, int c, double& val) {
    const unsigned long long own = raw[r * W + c];
    if (own != R3D_EMPTY_U64) { val = bits_dbl(own); return true; }
    for (int dr = -2; dr <= 2; ++dr)
        for (int dc = -1; dc <= 1; ++dc) {
            const int r1 = r + dr, c1 = c + dc;
            if (r1 < 0 || r1 >= H || c1 < 0 || c1 >= W) continue;          // outside the image: ignored by the erosion
            const int q = r1 * W + c1;
            if (!(dil[q >> 5] & (1u << (q & 31)))) return false;
        }
    int neighbors = 0;
    double sum = 0.0;
    for (int dr = -2; dr <= 2; ++dr)
        for (int dc = -1; dc <= 1; ++dc) {
            const int r1 = r + dr, c1 = c + dc;
            if (r1 < 0 || r1 >= H || c1 < 0 || c1 >= W) continue;
            const unsigned long long v = raw[r1 * W + c1];
            if (v != R3D_EMPTY_U64) { neighbors += 1; sum = add(sum, bits_dbl(v)); }
        }
    if (neighbors == 0) return false;
    val = mean_div(sum, neighbors);
    return true;
}

__device__ void bitonic_sort_u64(unsigned long long* keys, int n_pow2) {
    for (int k = 2; k <= n_pow2; k <<= 1)
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < n_pow2; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], bb = keys[ixj];
                    const bool up = (i & k) == 0;
                    if ((a > bb) == up) { keys[i] = bb; keys[ixj] = a; }
                }
            }
            __syncthreads();
        }
}

// A11 + A12 for the chosen candidate of each scan: the first feasible rotation that keeps >= min_points (accepted),
// else the last feasible one (its vis_px still deletes scene points in the reference, od/ins:472-501).  Builds the
// candidate's z-buffer in a scratch image, closes / fills it around the object, compares with the scene image
// (strict <) into the vis_px bit mask, and on acceptance appends the visible object points in (pix_id, index) order
// to the scene tail, the `check` record and the scene boxes.
#ifndef R3D_SEL_TILE_PX
#define R3D_SEL_TILE_PX 8192
#endif
constexpr int SEL_TILE_PX = R3D_SEL_TILE_PX;      // pixels of the shared-memory object tile (8 B of fp64 range each)

// local variant of obj_pixel_value on the shared-memory tile (rows r_lo.., cols c_lo.., nr x nc).  Pixels outside the
// tile but inside the image hold no object point and are farther than the 5x3 window from every object pixel, so
// their occupancy and dilation are 0; pixels outside the image are ignored by the erosion.
__device__ __forceinline__ bool tile_pixel_value(const unsigned long long* tile, const unsigned* dil, int H, int W, int r_lo,
                                                 int c_lo, int nr, int nc, int r, int c, double& val) {
    const unsigned long long own = tile[(r - r_lo) * nc + (c - c_lo)];
    if (own != R3D_EMPTY_U64) { val = bits_dbl(own); return true; }
    for (int dr = -2; dr <= 2; ++dr)
        for (int dc = -1; dc <= 1; ++dc) {
            const int r1 = r + dr, c1 = c + dc;
            if (r1 < 0 || r1 >= H || c1 < 0 || c1 >= W) continue;
            const int lr = r1 - r_lo, lc = c1 - c_lo;
            if (lr < 0 || lr >= nr || lc < 0 || lc >= nc) return false;
            const int q = lr * nc + lc;
            if (!(dil[q >> 5] & (1u << (q & 31)))) return false;
        }
    int neighbors = 0;
    double sum = 0.0;
    for (int dr = -2; dr <= 2; ++dr)
        for (int dc = -1; dc <= 1; ++dc) {
            const int lr = r + dr - r_lo, lc = c + dc - c_lo;
            if (lr < 0 || lr >= nr || lc < 0 || lc >= nc) continue;
            const unsigned long long v = tile[lr * nc + lc];
            if (v != R3D_EMPTY_U64) { neighbors += 1; sum = add(sum, bits_dbl(v)); }
        }
    if (neighbors == 0) return false;
    val = mean_div(sum, neighbors);
    return true;
}

// A11 + A12 for the chosen candidate of each scan: the first feasible rotation that keeps >= min_points (accepted),
// else the last feasible one (its vis_px still deletes scene points in the reference, od/ins:472-501).  Builds the
// candidate's z-buffer (in a shared-memory tile around the object when it fits, else in a global scratch image),
// closes / fills it, compares with the scene image (strict <) into the vis_px bit mask, and on acceptance appends the
// visible object points in (pix_id, index) order to the scene tail, the `check` record and the scene boxes.
// shared-memory scratch of the candidate selection: sort keys, ranges, object tile, pixel ids, dilation + visibility bits
struct SelScratch {
    unsigned long long* keys;      // [next_pow2(pts)]
    double* r;                     // [pts]
    unsigned long long* tile;      // [tile_px]
    int* pix;                      // [pts]
    unsigned *dil, *vis;           // [tile_px / 32] each
    int pts, tile_px;              // capacities (objects with more points / wider pixel rectangles use global scratch)
};
__device__ __forceinline__ SelScratch sel_scratch(unsigned long long* dyn, int key_cap, int pts, int tile_px) {
    SelScratch q;
    q.keys = dyn; q.r = reinterpret_cast<double*>(dyn + key_cap); q.tile = dyn + key_cap + pts;
    q.pix = reinterpret_cast<int*>(q.tile + tile_px); q.dil = reinterpret_cast<unsigned*>(q.pix + pts);
    q.vis = q.dil + tile_px / 32; q.pts = pts; q.tile_px = tile_px;
    return q;
}

// every thread of the CTA (any size) calls it; k = rotation of the chosen candidate, `accepted` = it keeps min_points
__device__ void select_emit_body(const EngineDev& e, int b, ScanState& s, int k, bool accepted, SelScratch q) {
    unsigned long long* s_keys = q.keys;
    double* s_r = q.r;
    unsigned long long* s_tile = q.tile;
    int* s_pix = q.pix;
    unsigned* s_dil = q.dil;
    unsigned* s_vis = q.vis;
    const int SEL_TILE_PX = q.tile_px;
    if (e.try_obj[b].count > q.pts) {
        s_keys = e.sel_keys + (size_t)b * e.sel_key_cap;
        s_r = e.sel_r + (size_t)b * e.max_obj_points;
        s_pix = e.sel_pix + (size_t)b * e.max_obj_points;
    }
    __shared__ int s_nvis;
    __shared__ int s_rect[4];
    __shared__ unsigned long long s_el[2];
    if (threadIdx.x == 0) {
        s_rect[0] = INT_MAX; s_rect[1] = -1; s_rect[2] = INT_MAX; s_rect[3] = -1; s_el[0] = R3D_EMPTY_U64; s_el[1] = 0ull;
        s_nvis = 0;
    }
    const ObjBox ob = e.obj[s.cur_obj];
    const ImageGeom g = s.geom;
    const int H = g.rows, W = g.cols;
    const size_t cb = (size_t)b * (e.K + 1);
    const double c = e.cos_k[k], sn = e.sin_k[k];
    const double level = e.cand_level[cb + k];
    const double dz = sub(level, ob.cz);
    unsigned* dm = e.dmask + (size_t)b * e.dwords;
    const double* smooth = e.smooth + (size_t)b * e.hw;
    const int t0 = s.n_tail, chk0 = s.n_check, nbox0 = s.n_boxes, nins0 = s.n_inserted, n0 = s.n0;
    // vis_px of the previous candidate lies inside the rectangle recorded with it: only those words are cleared (the
    // mask is all zero after a (re-)arm)
    if (s.d_r1 >= s.d_r0 && s.d_c1 >= s.d_c0) {
        const int nw = (s.d_c1 >> 5) - (s.d_c0 >> 5) + 2, nrow = s.d_r1 - s.d_r0 + 1;
        for (int i = threadIdx.x; i < nrow * nw; i += blockDim.x) {
            const int r = s.d_r0 + i / nw;
            const int w = ((r * e.cols + s.d_c0) >> 5) + i % nw;
            if (w <= ((r * e.cols + s.d_c1) >> 5)) dm[w] = 0u;
        }
    }
    __syncthreads();
    // project every object point once (od/ins:474-478); pixel rectangle of the object
    {
        int r_lo = INT_MAX, r_hi = -1, c_lo = INT_MAX, c_hi = -1;
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const ObjProj o = project_obj_point(e, ob, g, i, c, sn, dz, s);
            s_pix[i] = o.pix; s_r[i] = o.r;
            if (o.pix < 0) continue;
            const int pr = o.pix / W, pc = o.pix % W;
            r_lo = min(r_lo, pr); r_hi = max(r_hi, pr); c_lo = min(c_lo, pc); c_hi = max(c_hi, pc);
        }
        for (int o = 16; o > 0; o >>= 1) {
            r_lo = min(r_lo, __shfl_xor_sync(0xffffffffu, r_lo, o)); r_hi = max(r_hi, __shfl_xor_sync(0xffffffffu, r_hi, o));
            c_lo = min(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, o)); c_hi = max(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&s_rect[0], r_lo); atomicMax(&s_rect[1], r_hi); atomicMin(&s_rect[2], c_lo); atomicMax(&s_rect[3], c_hi);
        }
    }
    __syncthreads();
    const bool any_px = s_rect[1] >= 0;
    // vis_px can only lie within the object's pixels grown by the 5x3 window
    const int wr0 = any_px ? max(s_rect[0] - 2, 0) : 0, wr1 = any_px ? min(s_rect[1] + 2, H - 1) : -1;
    const int wc0 = any_px ? max(s_rect[2] - 1, 0) : 0, wc1 = any_px ? min(s_rect[3] + 1, W - 1) : -1;
    const int nr = wr1 - wr0 + 1, nc = wc1 - wc0 + 1;
    const bool in_smem = any_px && nr * nc <= SEL_TILE_PX;
    if (threadIdx.x == 0 && any_px) atomicAdd(&e.stats[in_smem ? 4 : 5], 1ull);
    if (in_smem) {
        const int npx = nr * nc;
        for (int i = threadIdx.x; i < npx; i += blockDim.x) s_tile[i] = R3D_EMPTY_U64;
        for (int i = threadIdx.x; i < (npx + 31) / 32; i += blockDim.x) { s_dil[i] = 0u; s_vis[i] = 0u; }
        __syncthreads();
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const int pix = s_pix[i];
            if (pix < 0) continue;
            const int pr = pix / W, pc = pix % W;
            atomicMin(&s_tile[(pr - wr0) * nc + (pc - wc0)], dbl_bits(s_r[i]));
            for (int dr = -2; dr <= 2; ++dr)                             // dilated occupancy (5 rows x 3 cols)
                for (int dc = -1; dc <= 1; ++dc) {
                    const int r1 = pr + dr, c1 = pc + dc;
                    if (r1 < 0 || r1 >= H || c1 < 0 || c1 >= W) continue;
                    const int q = (r1 - wr0) * nc + (c1 - wc0);
                    atomicOr(&s_dil[q >> 5], 1u << (q & 31));
                }
        }
        __syncthreads();
        // Only a pixel inside the dilated occupancy can survive the closing, and the dilation bits cover exactly the
        // 5x3 neighbourhoods of the object's pixels: one visit per such pixel of the tile (instead of one per
        // (object point, neighbour) pair, which evaluated most pixels many times).
        for (int lq = threadIdx.x; lq < npx; lq += blockDim.x) {
            if (!(s_dil[lq >> 5] & (1u << (lq & 31)))) continue;
            const int r = wr0 + lq / nc, cc = wc0 + lq % nc;
            double val;
            if (tile_pixel_value(s_tile, s_dil, H, W, wr0, wc0, nr, nc, r, cc, val) && val < smooth[r * W + cc]) {   // od/ins:486
                atomicOr(&s_vis[lq >> 5], 1u << (lq & 31));
                const int q = r * W + cc;
                atomicOr(&dm[q >> 5], 1u << (q & 31));
            }
        }
        __syncthreads();
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const int pix = s_pix[i];
            if (pix < 0) continue;
            const int lq = (pix / W - wr0) * nc + (pix % W - wc0);
            if (s_vis[lq >> 5] & (1u << (lq & 31))) {
                const int slot = atomicAdd(&s_nvis, 1);
                s_keys[slot] = ((unsigned long long)(unsigned)pix << 32) | (unsigned)i;
            }
        }
    } else if (any_px) {
        // object too wide for the tile (very close / very large): global scratch image + global dilation mask
        unsigned long long* raw = e.obj_raw + (size_t)b * e.hw;
        unsigned* vm = e.vmask + (size_t)b * e.dwords;
        for (int i = threadIdx.x; i < e.dwords; i += blockDim.x) vm[i] = 0u;
        __syncthreads();
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const int pix = s_pix[i];
            if (pix < 0) continue;
            atomicMin(&raw[pix], dbl_bits(s_r[i]));
            const int pr = pix / W, pc = pix % W;
            for (int dr = -2; dr <= 2; ++dr)
                for (int dc = -1; dc <= 1; ++dc) {
                    const int r1 = pr + dr, c1 = pc + dc;
                    if (r1 < 0 || r1 >= H || c1 < 0 || c1 >= W) continue;
                    const int q = r1 * W + c1;
                    atomicOr(&vm[q >> 5], 1u << (q & 31));
                }
        }
        __threadfence_block();
        __syncthreads();
        for (int t = threadIdx.x; t < ob.count * 15; t += blockDim.x) {
            const int i = t / 15, o = t % 15;
            const int pix = s_pix[i];
            if (pix < 0) continue;
            const int r = pix / W + (o / 3 - 2), cc = pix % W + (o % 3 - 1);
            if (r < 0 || r >= H || cc < 0 || cc >= W) continue;
            const int q = r * W + cc;
            double val;
            if (obj_pixel_value(raw, vm, H, W, r, cc, val) && val < smooth[q]) atomicOr(&dm[q >> 5], 1u << (q & 31));   // od/ins:486
        }
        __threadfence_block();
        __syncthreads();
        for (int i = threadIdx.x; i < ob.count; i += blockDim.x) {
            const int pix = s_pix[i];
            if (pix >= 0 && (dm[pix >> 5] & (1u << (pix & 31)))) {
                const int slot = atomicAdd(&s_nvis, 1);
                s_keys[slot] = ((unsigned long long)(unsigned)pix << 32) | (unsigned)i;
            }
            if (pix >= 0) raw[pix] = R3D_EMPTY_U64;                      // leave the scratch z-buffer empty
        }
    }
    __syncthreads();
    // visible object points, ordered by (pix_id, original index) as the reference's per-pixel loop emits them
    const int nvis = s_nvis;
    if (accepted) {
        if (e.try_obj[b].count <= q.pts) {
            // keys in shared memory: rank sort (the keys are distinct; one barrier instead of the log^2 barriers of the
            // bitonic network), the ordered keys go to the range scratch, which is free by now
            unsigned long long* sorted = reinterpret_cast<unsigned long long*>(s_r);
            for (int j = threadIdx.x; j < nvis; j += blockDim.x) {
                const unsigned long long key = s_keys[j];
                int rank = 0;
                for (int i = 0; i < nvis; ++i) rank += s_keys[i] < key;
                sorted[rank] = key;
            }
            __syncthreads();
            s_keys = sorted;
        } else {
            int np2 = 1;
            while (np2 < nvis) np2 <<= 1;
            for (int i = nvis + threadIdx.x; i < np2; i += blockDim.x) s_keys[i] = R3D_EMPTY_U64;
            __syncthreads();
            bitonic_sort_u64(s_keys, np2);
        }
        if (t0 + nvis > e.max_inserted || nbox0 + 1 > e.max_boxes || nins0 + 1 > e.max_events) {
            __syncthreads();
            if (threadIdx.x == 0) { set_error(s, R3D_ERR_CAPACITY); s.phase = PH_ERROR; }
        } else {
            const size_t base = (size_t)b * e.P + n0 + t0;
            const size_t tb = (size_t)b * e.max_inserted + t0;
            const size_t chk = ((size_t)b * e.max_inserted + chk0) * 5;
            for (int j = threadIdx.x; j < nvis; j += blockDim.x) {
                const int i = (int)(s_keys[j] & 0xffffffffull);
                const ObjProj o = project_obj_point(e, ob, g, i, c, sn, dz, s);
                e.tail_x[tb + j] = o.x; e.tail_y[tb + j] = o.y; e.tail_z[tb + j] = o.z;
                const float inten = e.obj_i[ob.first + i];
                const unsigned lab = e.obj_label[ob.first + i];
                e.tail_i[tb + j] = inten;
                e.label[base + j] = lab;
                e.r[base + j] = o.r; e.el[base + j] = o.el;
                atomicMin(&s_el[0], dbl_bits(o.el)); atomicMax(&s_el[1], dbl_bits(o.el));
                e.col[base + j] = (unsigned short)o.col;
                e.pix[base + j] = o.pix;
                e.alive[base + j] = 1;
                float* ck = e.check + chk + (size_t)j * 5;
                ck[0] = (float)o.x; ck[1] = (float)o.y; ck[2] = (float)o.z; ck[3] = inten; ck[4] = (float)lab;
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                int* rec = e.inserted + ((size_t)b * e.max_events + nins0) * 4;
                rec[0] = s.cur_obj; rec[1] = k; rec[2] = ob.cls; rec[3] = nvis;
                const YawBox yb = make_yaw_box(ob.cx, ob.cy, ob.a, ob.b, c, sn);
                double* ib = e.inserted_box + ((size_t)b * e.max_events + nins0) * 8;
                ib[0] = yb.cx; ib[1] = yb.cy; ib[2] = level; ib[3] = yb.m00; ib[4] = yb.m10;
                ib[5] = ob.length; ib[6] = ob.width; ib[7] = ob.height;
                Box bx = yaw_box_to_box(yb, level, ob.length, ob.width, ob.height);      // od/ins:555
                bx.reach = ob.reach;
                e.boxes[(size_t)b * e.max_boxes + nbox0] = bx;
                e.box_tests[(size_t)b * e.max_boxes + nbox0] = make_box_test(bx);
                s.n_boxes = nbox0 + 1; s.n_inserted = nins0 + 1;
                s.tail_before = t0; s.n_tail = t0 + nvis; s.n_check = chk0 + nvis;
                s.new_min_bits = s_el[0]; s.new_max_bits = s_el[1];
            }
        }
    }
    if (threadIdx.x == 0) {
        s.accepted = accepted ? 1 : 0; s.chosen_rot = k; s.chosen_v = nvis;
        s.d_r0 = wr0; s.d_r1 = wr1; s.d_c0 = wc0; s.d_c1 = wc1;
        if (!accepted) { s.new_min_bits = R3D_EMPTY_U64; s.new_max_bits = 0ull; }
    }
}

__global__ void __launch_bounds__(512) k_select_emit(EngineDev e, int n_scans, int key_cap, int smem_pts) {
    const int b = blockIdx.x;
    if (b >= n_scans || !e.gate_try[b]) return;
    ScanState& s = e.st[b];
    const int nf = s.n_feasible;
    if (nf == 0) return;
    extern __shared__ unsigned long long s_dyn[];
    const bool accepted = s.found_rank < nf;
    const int rank = accepted ? s.found_rank : nf - 1;
    select_emit_body(e, b, s, e.feas[(size_t)b * e.K + rank], accepted, sel_scratch(s_dyn, key_cap, smem_pts, SEL_TILE_PX));
}
