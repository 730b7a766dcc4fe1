// A4: class_closing + smooth_out (cl:9-62) as one tiled stencil kernel.
//   closing(rectangle(5, 3)) = 5 rows x 3 cols dilate then erode on the binary occupancy, pixels outside the image
//   ignored, no azimuth wrap; pixels switched on by the closing that hold no point get the mean of their occupied
//   neighbours' ORIGINAL ranges, summed in the reference's (drow, dcol) order in fp64 (cl:46-51,57).
// Templated on the input adaptor so the same code serves the float64 train/label pair of the drop-in smooth_out and
// the engine's raw uint64 z-buffer.  The tile (+ a 4-row / 2-col halo) is staged once in shared memory with
// coalesced row reads; dilation, erosion and the hole fill then run out of shared memory, so HBM sees one read of
// the input (x1.33 for the halo, mostly L2 hits) and one write of the output: 16 B/pixel for the engine variant.
#pragma once
#include <cuda.h>            // CUtensorMap (the TMA descriptor of the z-buffer; encoded through the driver entry point)
#include "r3d_common.cuh"

constexpr int CF_TH = 32;       // output rows per CTA
constexpr int CF_TW = 64;       // output cols per CTA
constexpr int CF_THREADS = 256;
constexpr int CF_HR = 4, CF_HC = 2;                    // halo: two 5x3 passes
constexpr int CF_SH = CF_TH + 2 * CF_HR;               // staged rows
constexpr int CF_SW = CF_TW + 2 * CF_HC;               // staged cols

// one CF_TH x CF_TW output tile at (r0, c0) of image z; every thread of the CTA calls it (it synchronises).
// The binary morphology runs on BIT ROWS: a staged row of 68 pixels is three 32-bit words built with one warp ballot
// per 32 pixels while the values are staged; the 5 x 3 dilation / erosion are a handful of shifts and ORs / ANDs per
// row word (out-of-image positions: occupancy 0, dilation 1 = neutral for the erosion), so the per-pixel work that
// remains is the ordered fp64 neighbour mean of the pixels the closing switched on.
constexpr int CF_WORDS = 4;                            // 68 staged columns -> 3 words (+ 1 zero word for the funnel shifts)
template <class In>
__device__ __forceinline__ void close_fill_tile(const In& in, int H, int W, int64_t base, int r0, int c0, int z,
                                                double* __restrict__ out_train, double* __restrict__ out_label,
                                                uint8_t* __restrict__ closed_out, int* __restrict__ far_flag) {
    __shared__ double s_val[CF_SH][CF_SW];
    __shared__ unsigned s_occ[CF_SH][CF_WORDS];        // clip(label, 0, 1) > 0
    __shared__ unsigned s_one[CF_SH][CF_WORDS];        // label == 1
    __shared__ unsigned s_in[CF_SH][CF_WORDS];         // inside the image
    __shared__ unsigned s_dil[CF_SH][CF_WORDS];
    __shared__ unsigned s_ero[CF_SH][CF_WORDS];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    // (row, word) units, one warp each: all loads of a warp are issued before the first ballot waits for one
    constexpr int UNITS = CF_SH * 3, PER_WARP = UNITS / (CF_THREADS / 32);
    static_assert(UNITS % (CF_THREADS / 32) == 0, "close/fill staging: units must divide evenly over the warps");
    constexpr int BATCH = 5;                           // loads in flight per lane
    static_assert(PER_WARP % BATCH == 0, "close/fill staging: batches must divide the units of a warp");
    for (int k0 = 0; k0 < PER_WARP; k0 += BATCH) {
        double v[BATCH];
        uint8_t o[BATCH];
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
            const int u = warp + (k0 + k) * (CF_THREADS / 32), lr = u / 3, lc = (u % 3) * 32 + lane;
            const int r = r0 - CF_HR + lr, c = c0 - CF_HC + lc;
            v[k] = 0.0; o[k] = 0;
            if (lc < CF_SW && r >= 0 && r < H && c >= 0 && c < W) { in.load(base + (int64_t)r * W + c, v[k], o[k]); o[k] |= 4; }
        }
#pragma unroll
        for (int k = 0; k < BATCH; ++k) {
            const int u = warp + (k0 + k) * (CF_THREADS / 32), lr = u / 3, w = u % 3, lc = w * 32 + lane;
            if (lc < CF_SW) s_val[lr][lc] = v[k];
            const unsigned b_occ = __ballot_sync(0xffffffffu, o[k] & 1), b_one = __ballot_sync(0xffffffffu, o[k] & 2);
            const unsigned b_in = __ballot_sync(0xffffffffu, o[k] & 4);
            if (lane == 0) { s_occ[lr][w] = b_occ; s_one[lr][w] = b_one; s_in[lr][w] = b_in; }
        }
    }
    if (threadIdx.x < CF_SH) { s_occ[threadIdx.x][3] = 0u; s_one[threadIdx.x][3] = 0u; s_in[threadIdx.x][3] = 0u; }
    __syncthreads();
    // horizontal 3-window of a bit row: bit c <- f(c - 1, c, c + 1), shifts carried across the words
    auto left = [](const unsigned* a, int w) { return (a[w] << 1) | (w > 0 ? a[w - 1] >> 31 : 0u); };
    auto right = [](const unsigned* a, int w) { return (a[w] >> 1) | (a[w + 1] << 31); };
    if (threadIdx.x < (CF_SH - 4) * 3) {               // dilation, staged rows 2 .. CF_SH - 3
        const int lr = 2 + threadIdx.x / 3, w = threadIdx.x % 3;
        unsigned d = 0u;
#pragma unroll
        for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = s_occ[lr + dr]; d |= a[w] | left(a, w) | right(a, w); }
        s_dil[lr][w] = d | ~s_in[lr][w];               // outside the image: neutral for the erosion
    }
    if (threadIdx.x < CF_SH) s_dil[threadIdx.x][3] = ~0u;
    __syncthreads();
    if (threadIdx.x < CF_TH * 3) {                     // erosion, staged rows 4 .. CF_SH - 5 (the output rows)
        const int lr = CF_HR + threadIdx.x / 3, w = threadIdx.x % 3;
        unsigned e = ~0u;
#pragma unroll
        for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = s_dil[lr + dr]; e &= a[w] & left(a, w) & right(a, w); }
        s_ero[lr][w] = e;
    }
    __syncthreads();
    bool far = false;
    for (int i = threadIdx.x; i < CF_TH * CF_TW; i += CF_THREADS) {
        const int lr = i / CF_TW, lc = i % CF_TW;
        const int r = r0 + lr, c = c0 + lc;
        if (r >= H || c >= W) continue;
        const int sr = lr + CF_HR, sc = lc + CF_HC;
        const bool e = (s_ero[sr][sc >> 5] >> (sc & 31)) & 1u;
        const bool one = (s_one[sr][sc >> 5] >> (sc & 31)) & 1u;
        double t = s_val[sr][sc];
        bool filled = false;
        if (e && !one) {                                  // cl:41-43: closed == 255 and label != 1
            int neighbors = 0;
            double sum = 0.0;
            const int q = sc - 1, qw = q >> 5, qb = q & 31;
#pragma unroll
            for (int dr = -2; dr <= 2; ++dr) {             // cl:46-51: (drow, dcol) order; out-of-image neighbours are "not 1"
                const unsigned m = __funnelshift_r(s_one[sr + dr][qw], s_one[sr + dr][qw + 1], qb) & 7u;
                if (m & 1u) { neighbors += 1; sum = r3d::add(sum, s_val[sr + dr][sc - 1]); }
                if (m & 2u) { neighbors += 1; sum = r3d::add(sum, s_val[sr + dr][sc]); }
                if (m & 4u) { neighbors += 1; sum = r3d::add(sum, s_val[sr + dr][sc + 1]); }
            }
            if (neighbors > 0) t = r3d::mean_div(sum, neighbors);        // cl:57
            filled = true;                                                   // cl:55,58: label = 1
        }
        const int64_t idx = base + (int64_t)r * W + c;
        out_train[idx] = t;
        if (out_label) out_label[idx] = filled ? 1.0 : in.lab(idx);
        if (closed_out) closed_out[idx] = e ? 255 : 0;
        far |= t > r3d::kEmptyRange;
    }
    if (far_flag && far) atomicOr(&far_flag[z], 1);
}

// one image per blockIdx.z, tiles on the (x, y) grid
template <class In>
__global__ void __launch_bounds__(CF_THREADS) k_close_fill(In in, int H, int W, int64_t img_stride,
                                                            double* __restrict__ out_train, double* __restrict__ out_label,
                                                            uint8_t* __restrict__ closed_out, int* __restrict__ far_flag) {
    const int z = blockIdx.z;
    close_fill_tile(in, H, W, (int64_t)z * img_stride, (int)blockIdx.y * CF_TH, (int)blockIdx.x * CF_TW, z, out_train, out_label,
                    closed_out, far_flag);
}

// the engine's variant: a persistent grid walks the (image, tile) tasks k_update listed for this round — after the
// first round only the few tiles around an inserted object change, so a grid over every tile of every image would be
// tens of thousands of CTAs that exit at once.  task = image * tiles_per_image + tile.
template <class In>
__global__ void __launch_bounds__(CF_THREADS, 4) k_close_fill_tasks(In in, int H, int W, int64_t img_stride,
                                                                  double* __restrict__ out_train, int* __restrict__ far_flag,
                                                                  const int* __restrict__ tasks, const int* __restrict__ n_tasks) {
    const int tiles_x = (W + CF_TW - 1) / CF_TW, tiles = tiles_x * ((H + CF_TH - 1) / CF_TH);
    const int n = *n_tasks;
    for (int t = blockIdx.x; t < n; t += gridDim.x) {
        const int task = tasks[t], z = task / tiles, tile = task % tiles;
        close_fill_tile(in, H, W, (int64_t)z * img_stride, (tile / tiles_x) * CF_TH, (tile % tiles_x) * CF_TW, z, out_train,
                        (double*)nullptr, (uint8_t*)nullptr, far_flag);
        __syncthreads();                                 // the tile buffers are reused by the next task
    }
}

// The engine's z-buffer variant, software pipelined: while a CTA closes / fills one tile out of shared memory, the raw
// 64-bit range words of its NEXT task are already on their way (cp.async, 16 bytes per request, double buffered), so
// the HBM latency of a tile is hidden behind the work on the previous one instead of being paid once per tile.
// Needs an even image width (16-byte aligned row segments); the launch falls back to k_close_fill_tasks otherwise.
static __device__ __forceinline__ void cf_async_copy16(void* smem, const void* gmem) {
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem) : "memory");
}
// shared memory of the pipelined walk: two raw tiles + four bit-row images
struct CfPipeSmem {
    unsigned long long raw[2][CF_SH][CF_SW];
    unsigned one[CF_SH][CF_WORDS], in[CF_SH][CF_WORDS], dil[CF_SH][CF_WORDS], ero[CF_SH][CF_WORDS];
};
// tasks t0, t0 + tstep, ... < n of a CTA of NT threads; task_of(t) = image * tiles_per_image + tile
template <int NT, class TaskOf>
static __device__ __forceinline__ void cf_pipelined_tiles(CfPipeSmem& sm, const unsigned long long* __restrict__ raw, int H, int W,
                                                          int64_t img_stride, double* __restrict__ out_train, int* __restrict__ far_flag,
                                                          int t0, int n, int tstep, TaskOf task_of) {
    const int tiles_x = (W + CF_TW - 1) / CF_TW, tiles = tiles_x * ((H + CF_TH - 1) / CF_TH);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    constexpr int CHUNKS = CF_SW / 2;                  // 16-byte requests per staged row
    auto issue = [&](int t, int buf) {
        const int task = task_of(t), z = task / tiles, tile = task % tiles;
        const int r0 = (tile / tiles_x) * CF_TH, c0 = (tile % tiles_x) * CF_TW;
        const unsigned long long* img = raw + (int64_t)z * img_stride;
        for (int i = threadIdx.x; i < CF_SH * CHUNKS; i += NT) {
            const int lr = i / CHUNKS, ch = i % CHUNKS;
            const int r = r0 - CF_HR + lr, c = c0 - CF_HC + 2 * ch;
            if (r >= 0 && r < H && c >= 0 && c + 1 < W) cf_async_copy16(&sm.raw[buf][lr][2 * ch], img + (int64_t)r * W + c);
        }
    };
    auto left = [](const unsigned* a, int w) { return (a[w] << 1) | (w > 0 ? a[w - 1] >> 31 : 0u); };
    auto right = [](const unsigned* a, int w) { return (a[w] >> 1) | (a[w + 1] << 31); };
    int t = t0;
    if (t < n) issue(t, 0);
    asm volatile("cp.async.commit_group;" ::: "memory");
    if (threadIdx.x < CF_SH) { sm.one[threadIdx.x][3] = 0u; sm.in[threadIdx.x][3] = 0u; sm.dil[threadIdx.x][3] = ~0u; }
    for (int buf = 0; t < n; t += tstep, buf ^= 1) {
        if (t + tstep < n) issue(t + tstep, buf ^ 1);
        asm volatile("cp.async.commit_group;" ::: "memory");
        asm volatile("cp.async.wait_group 1;" ::: "memory");          // everything but the newest group has landed
        __syncthreads();
        const int task = task_of(t), z = task / tiles, tile = task % tiles;
        const int r0 = (tile / tiles_x) * CF_TH, c0 = (tile % tiles_x) * CF_TW;
        const int64_t base = (int64_t)z * img_stride;
        for (int u = warp; u < CF_SH * 3; u += NT / 32) {             // bit rows of the staged tile
            const int lr = u / 3, w = u % 3, lc = w * 32 + lane;
            const int r = r0 - CF_HR + lr, c = c0 - CF_HC + lc;
            const bool inside = lc < CF_SW && r >= 0 && r < H && c >= 0 && c < W;
            const bool hit = inside && sm.raw[buf][lr][min(lc, CF_SW - 1)] != R3D_EMPTY_U64;
            const unsigned b_one = __ballot_sync(0xffffffffu, hit), b_in = __ballot_sync(0xffffffffu, inside);
            if (lane == 0) { sm.one[lr][w] = b_one; sm.in[lr][w] = b_in; }
        }
        __syncthreads();
        if (threadIdx.x < (CF_SH - 4) * 3) {
            const int lr = 2 + threadIdx.x / 3, w = threadIdx.x % 3;
            unsigned d = 0u;
#pragma unroll
            for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = sm.one[lr + dr]; d |= a[w] | left(a, w) | right(a, w); }
            sm.dil[lr][w] = d | ~sm.in[lr][w];
        }
        __syncthreads();
        if (threadIdx.x < CF_TH * 3) {
            const int lr = CF_HR + threadIdx.x / 3, w = threadIdx.x % 3;
            unsigned e = ~0u;
#pragma unroll
            for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = sm.dil[lr + dr]; e &= a[w] & left(a, w) & right(a, w); }
            sm.ero[lr][w] = e;
        }
        __syncthreads();
        bool far = false;
        for (int i = threadIdx.x; i < CF_TH * CF_TW; i += NT) {
            const int lr = i / CF_TW, lc = i % CF_TW;
            const int r = r0 + lr, c = c0 + lc;
            if (r >= H || c >= W) continue;
            const int sr = lr + CF_HR, sc = lc + CF_HC;
            const bool e = (sm.ero[sr][sc >> 5] >> (sc & 31)) & 1u;
            const bool one = (sm.one[sr][sc >> 5] >> (sc & 31)) & 1u;
            double tv = one ? r3d::bits_dbl(sm.raw[buf][sr][sc]) : r3d::kEmptyRange;      // od/ins:100: empty = 500
            if (e && !one) {                                  // cl:41-43
                int neighbors = 0;
                double sum = 0.0;
                const int q = sc - 1, qw = q >> 5, qb = q & 31;
#pragma unroll
                for (int dr = -2; dr <= 2; ++dr) {             // cl:46-51, (drow, dcol) order
                    const unsigned m = __funnelshift_r(sm.one[sr + dr][qw], sm.one[sr + dr][qw + 1], qb) & 7u;
                    if (m & 1u) { neighbors += 1; sum = r3d::add(sum, r3d::bits_dbl(sm.raw[buf][sr + dr][sc - 1])); }
                    if (m & 2u) { neighbors += 1; sum = r3d::add(sum, r3d::bits_dbl(sm.raw[buf][sr + dr][sc])); }
                    if (m & 4u) { neighbors += 1; sum = r3d::add(sum, r3d::bits_dbl(sm.raw[buf][sr + dr][sc + 1])); }
                }
                if (neighbors > 0) tv = r3d::mean_div(sum, neighbors);       // cl:57
            }
            out_train[base + (int64_t)r * W + c] = tv;
            far |= tv > r3d::kEmptyRange;
        }
        if (far) atomicOr(&far_flag[z], 1);
        __syncthreads();                                  // sm.raw[buf] is the target of the loads issued two tasks ahead
    }
}
static __global__ void __launch_bounds__(CF_THREADS, 4) k_close_fill_raw_pipelined(const unsigned long long* __restrict__ raw, int H, int W,
                                                                           int64_t img_stride, double* __restrict__ out_train,
                                                                           int* __restrict__ far_flag, const int* __restrict__ tasks,
                                                                           const int* __restrict__ n_tasks) {
    __shared__ __align__(16) CfPipeSmem sm;
    cf_pipelined_tiles<CF_THREADS>(sm, raw, H, W, img_stride, out_train, far_flag, (int)blockIdx.x, *n_tasks, (int)gridDim.x,
                                   [&](int t) { return tasks[t]; });
}


// ---- the same walk with the tile loads done by the TMA unit (sm_90+; here sm_100a): ONE thread arms an mbarrier with
// the byte count of a staged tile and issues one `cp.async.bulk.tensor.3d` for the 68 x 40 x 1 box at
// (c0 - 2, r0 - 4, image) of the [B][H][W] u64 z-buffer; the unit does the address arithmetic and fills whatever lies
// outside the image with zeros.  A range of 0.0 cannot occur (r > 0 is asserted at ingest), so "0" doubles as the
// outside marker and the per-pixel border tests of the cp.async variant disappear; the CTA waits on the mbarrier phase
// instead of `cp.async.wait_group` + barrier.  Double buffered like the variant above.
static __device__ __forceinline__ unsigned cf_smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
static __device__ __forceinline__ void cf_mbar_init(unsigned long long* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(cf_smem_u32(bar)), "r"(count) : "memory");
}
static __device__ __forceinline__ void cf_mbar_expect_tx(unsigned long long* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(cf_smem_u32(bar)), "r"(bytes) : "memory");
}
static __device__ __forceinline__ void cf_mbar_wait(unsigned long long* bar, unsigned phase) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "CF_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra CF_DONE;\n"
        "bra CF_WAIT;\n"
        "CF_DONE:\n"
        "}" ::"r"(cf_smem_u32(bar)), "r"(phase) : "memory");
}
static __device__ __forceinline__ void cf_tma_load_3d(void* dst, const CUtensorMap* tm, unsigned long long* bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(cf_smem_u32(dst)), "l"(tm), "r"(cf_smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
static __global__ void __launch_bounds__(CF_THREADS, 4) k_close_fill_tma(const __grid_constant__ CUtensorMap tmap, int H, int W, int64_t img_stride,
                                                                         double* __restrict__ out_train, int* __restrict__ far_flag,
                                                                         const int* __restrict__ tasks, const int* __restrict__ n_tasks) {
    __shared__ __align__(128) unsigned long long s_raw[2][CF_SH][CF_SW];
    __shared__ unsigned s_one[CF_SH][CF_WORDS], s_in[CF_SH][CF_WORDS], s_dil[CF_SH][CF_WORDS], s_ero[CF_SH][CF_WORDS];
    __shared__ __align__(8) unsigned long long s_bar[2];
    const int tiles_x = (W + CF_TW - 1) / CF_TW, tiles = tiles_x * ((H + CF_TH - 1) / CF_TH);
    const int n = *n_tasks;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) {
        cf_mbar_init(&s_bar[0], 1); cf_mbar_init(&s_bar[1], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    if (threadIdx.x < CF_SH) { s_one[threadIdx.x][3] = 0u; s_in[threadIdx.x][3] = 0u; s_dil[threadIdx.x][3] = ~0u; s_ero[threadIdx.x][3] = 0u; }
    __syncthreads();
    auto issue = [&](int t, int buf) {                 // one thread
        const int task = tasks[t], z = task / tiles, tile = task % tiles;
        cf_mbar_expect_tx(&s_bar[buf], (unsigned)(CF_SH * CF_SW * sizeof(unsigned long long)));
        cf_tma_load_3d(&s_raw[buf][0][0], &tmap, &s_bar[buf], (tile % tiles_x) * CF_TW - CF_HC, (tile / tiles_x) * CF_TH - CF_HR, z);
    };
    auto left = [](const unsigned* a, int w) { return (a[w] << 1) | (w > 0 ? a[w - 1] >> 31 : 0u); };
    auto right = [](const unsigned* a, int w) { return (a[w] >> 1) | (a[w + 1] << 31); };
    int t = blockIdx.x;
    unsigned phases = 0u;                              // bit b = parity the next wait on buffer b looks for
    if (t < n && threadIdx.x == 0) issue(t, 0);
    for (int buf = 0; t < n; t += gridDim.x, buf ^= 1) {
        if (threadIdx.x == 0 && t + (int)gridDim.x < n) issue(t + gridDim.x, buf ^ 1);
        cf_mbar_wait(&s_bar[buf], (phases >> buf) & 1u);
        phases ^= 1u << buf;
        const int task = tasks[t], z = task / tiles, tile = task % tiles;
        const int r0 = (tile / tiles_x) * CF_TH, c0 = (tile % tiles_x) * CF_TW;
        const int64_t base = (int64_t)z * img_stride;
        for (int lr = warp; lr < CF_SH; lr += CF_THREADS / 32) {      // bit rows of the staged tile, one staged row per warp
            const unsigned long long v0 = s_raw[buf][lr][lane], v1 = s_raw[buf][lr][32 + lane];
            const unsigned long long v2 = lane < CF_SW - 64 ? s_raw[buf][lr][64 + lane] : 0ull;
            const unsigned i0 = __ballot_sync(0xffffffffu, v0 != 0ull), i1 = __ballot_sync(0xffffffffu, v1 != 0ull);
            const unsigned i2 = __ballot_sync(0xffffffffu, v2 != 0ull);
            const unsigned o0 = __ballot_sync(0xffffffffu, v0 != 0ull && v0 != R3D_EMPTY_U64);
            const unsigned o1 = __ballot_sync(0xffffffffu, v1 != 0ull && v1 != R3D_EMPTY_U64);
            const unsigned o2 = __ballot_sync(0xffffffffu, v2 != 0ull && v2 != R3D_EMPTY_U64);
            if (lane < 3) {
                s_one[lr][lane] = lane == 0 ? o0 : (lane == 1 ? o1 : o2);
                s_in[lr][lane] = lane == 0 ? i0 : (lane == 1 ? i1 : i2);
            }
        }
        __syncthreads();
        if (threadIdx.x < (CF_SH - 4) * 3) {
            const int lr = 2 + threadIdx.x / 3, w = threadIdx.x % 3;
            unsigned d = 0u;
#pragma unroll
            for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = s_one[lr + dr]; d |= a[w] | left(a, w) | right(a, w); }
            s_dil[lr][w] = d | ~s_in[lr][w];
        }
        __syncthreads();
        if (threadIdx.x < CF_TH * 3) {
            const int lr = CF_HR + threadIdx.x / 3, w = threadIdx.x % 3;
            unsigned e = ~0u;
#pragma unroll
            for (int dr = -2; dr <= 2; ++dr) { const unsigned* a = s_dil[lr + dr]; e &= a[w] & left(a, w) & right(a, w); }
            s_ero[lr][w] = e;
        }
        __syncthreads();
        bool far = false;
        // two horizontally adjacent output pixels per thread: their 5 x 3 neighbourhoods share two of three columns, so one
        // 4-bit window per row serves both, and the pair leaves as one 16-byte store (W is even with a tensor map)
        for (int i = threadIdx.x; i < CF_TH * CF_TW / 2; i += CF_THREADS) {
            const int lr = i / (CF_TW / 2), lc = (i % (CF_TW / 2)) * 2;
            const int r = r0 + lr, c = c0 + lc;
            if (r >= H || c >= W) continue;
            const int sr = lr + CF_HR, sc = lc + CF_HC;
            const int q = sc - 1, qw = q >> 5, qb = q & 31;                  // window bits: columns sc - 1 .. sc + 2
            const unsigned e2 = __funnelshift_r(s_ero[sr][sc >> 5], s_ero[sr][(sc >> 5) + 1], sc & 31) & 3u;
            unsigned win[5];
#pragma unroll
            for (int dr = -2; dr <= 2; ++dr) win[dr + 2] = __funnelshift_r(s_one[sr + dr][qw], s_one[sr + dr][qw + 1], qb) & 15u;
            double tv[2];
#pragma unroll
            for (int u = 0; u < 2; ++u) {
                const bool one = (win[2] >> (1 + u)) & 1u, e = (e2 >> u) & 1u;
                tv[u] = one ? r3d::bits_dbl(s_raw[buf][sr][sc + u]) : r3d::kEmptyRange;  // od/ins:100: empty = 500
                if (e && !one) {                                  // cl:41-43
                    int neighbors = 0;
                    double sum = 0.0;
#pragma unroll
                    for (int dr = -2; dr <= 2; ++dr) {             // cl:46-51, (drow, dcol) order
                        const unsigned m = (win[dr + 2] >> u) & 7u;
                        if (m & 1u) { neighbors += 1; sum = r3d::add(sum, r3d::bits_dbl(s_raw[buf][sr + dr][sc + u - 1])); }
                        if (m & 2u) { neighbors += 1; sum = r3d::add(sum, r3d::bits_dbl(s_raw[buf][sr + dr][sc + u])); }
                        if (m & 4u) { neighbors += 1; sum = r3d::add(sum, r3d::bits_dbl(s_raw[buf][sr + dr][sc + u + 1])); }
                    }
                    if (neighbors > 0) tv[u] = r3d::mean_div(sum, neighbors);    // cl:57
                }
                far |= tv[u] > r3d::kEmptyRange;
            }
            *reinterpret_cast<double2*>(out_train + base + (int64_t)r * W + c) = make_double2(tv[0], tv[1]);
        }
        if (far) atomicOr(&far_flag[z], 1);
        __syncthreads();                                  // s_raw[buf] is the target of the TMA load issued two tasks ahead
    }
}
