// Kernels of the batched Real3D-Aug engine, part: A14 output compaction.
// Included by r3d_engine_kernels.cuh (inside namespace r3d, after the shared constants); not a standalone header.
// --------------------------------------------------------------------------------------------- outputs
// A14 (od/ds:76-109, ss/ds:72-106): surviving rows in order (original points, then inserted points), cast to
// float32 / uint32.  40 B/point of algorithmic traffic.
// Three launches: per-chunk live counts (grid = chunks x scans), offsets (one CTA: totals per scan, exclusive scan over
// the scans, chunk offsets), chunk-wise stable compaction.
__global__ void __launch_bounds__(STREAM_THREADS) k_out_count(EngineDev e, int n_scans) {
    const int b = blockIdx.y;
    if (b >= n_scans) return;
    const ScanState& s = e.st[b];
    const int n = s.n0 + s.n_tail;
    const int p0 = blockIdx.x * CHUNK;
    const size_t base = (size_t)b * e.P;
    int cnt = 0;
    if (p0 < n) {
        const int p1 = min(p0 + CHUNK, n);
        if (p1 - p0 == CHUNK && ((base + p0) & 15) == 0) {     // whole aligned chunk: 16 alive bytes per thread in one load
            const uint4 v = *reinterpret_cast<const uint4*>(e.alive + base + p0 + threadIdx.x * 16);
            cnt = __popc(v.x & 0x01010101u) + __popc(v.y & 0x01010101u) + __popc(v.z & 0x01010101u) + __popc(v.w & 0x01010101u);
        } else {
            for (int p = p0 + threadIdx.x; p < p1; p += STREAM_THREADS) cnt += e.alive[base + p] ? 1 : 0;
        }
    }
    __shared__ int s_w[STREAM_THREADS / 32];
    for (int o = 16; o > 0; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < STREAM_THREADS / 32; ++w) t += s_w[w];
        e.chunk_cnt[(size_t)b * e.max_chunks + blockIdx.x] = t;
    }
}

__global__ void __launch_bounds__(1024) k_out_offsets(EngineDev e, int n_scans, int chunks) {
    __shared__ long long s_w[32], s_c[32];
    __shared__ long long s_run, s_crun;
    if (threadIdx.x == 0) { s_run = 0; s_crun = 0; }
    __syncthreads();
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    for (int b0 = 0; b0 < n_scans; b0 += 1024) {
        const int b = b0 + threadIdx.x;
        long long tot = 0, chk = 0;
        if (b < n_scans) {
            const int* cc = e.chunk_cnt + (size_t)b * e.max_chunks;
            for (int c = 0; c < chunks; ++c) tot += cc[c];
            chk = e.st[b].n_check;
        }
        long long inc = tot, cinc = chk;
        for (int o = 1; o < 32; o <<= 1) {
            const long long t = __shfl_up_sync(0xffffffffu, inc, o), u = __shfl_up_sync(0xffffffffu, cinc, o);
            if (lane >= o) { inc += t; cinc += u; }
        }
        if (lane == 31) { s_w[w] = inc; s_c[w] = cinc; }
        __syncthreads();
        long long off = s_run, coff = s_crun;
        for (int i = 0; i < w; ++i) { off += s_w[i]; coff += s_c[i]; }
        if (b < n_scans) {
            e.out_off[b] = off + inc - tot; e.check_off[b] = coff + cinc - chk; e.out_count[b] = tot;
            if (b == n_scans - 1) { e.out_off[n_scans] = off + inc; e.check_off[n_scans] = coff + cinc; }
        }
        __syncthreads();
        if (threadIdx.x == 1023) { s_run = off + inc; s_crun = coff + cinc; }
        __syncthreads();
    }
}

// WORLD: e.world is set and every output point and check row goes through the scan's world transform on its way out
// (no extra bytes); the instantiation without it is the plain compaction
template <bool WORLD>
__global__ void __launch_bounds__(STREAM_THREADS) k_out_write(EngineDev e, int n_scans) {
    const int b = blockIdx.y;
    if (b >= n_scans) return;
    const ScanState& s = e.st[b];
    const int n = s.n0 + s.n_tail;
    const int p0 = blockIdx.x * CHUNK;
    const size_t base = (size_t)b * e.P;
    [[maybe_unused]] WorldXf wx{};
    if constexpr (WORLD) wx = world_xf(e.world + (size_t)b * 8);
    if (blockIdx.x == 0) {                              // the `check` record of the scan (od/ds:91-93)
        const long long c0 = e.check_off[b];
        const float* ck = e.check + (size_t)b * e.max_inserted * 5;
        if constexpr (WORLD) {
            for (int r = threadIdx.x; r < s.n_check; r += blockDim.x) {
                const float* in = ck + (size_t)r * 5;
                float* out = e.out_check + (c0 + r) * 5;
                float x = in[0], y = in[1], z = in[2];
                world_point(wx, x, y, z);
                out[0] = x; out[1] = y; out[2] = z; out[3] = in[3]; out[4] = in[4];
            }
        } else {
            for (int i = threadIdx.x; i < s.n_check * 5; i += blockDim.x) e.out_check[c0 * 5 + i] = ck[i];
        }
    }
    if (p0 >= n) return;
    long long o0 = e.out_off[b];
    {
        const int* cc = e.chunk_cnt + (size_t)b * e.max_chunks;
        for (int c = 0; c < (int)blockIdx.x; ++c) o0 += cc[c];
    }
    // every warp owns a contiguous slice of the chunk (CHUNK / warps points): the live counts of the slices give the
    // warps their output offsets with ONE barrier, after which a warp compacts its slice 32 points at a time with
    // ballots only
    constexpr int NW = STREAM_THREADS / 32, SLICE = CHUNK / NW;
    static_assert(SLICE % 32 == 0 && SLICE / 32 <= 32, "one alive word per lane covers the slice");
    __shared__ int s_w[NW];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int q0 = p0 + w * SLICE, q1 = min(q0 + SLICE, n);
    int mine = 0;
    for (int p = q0 + lane; p < q1; p += 32) mine += e.alive[base + p] ? 1 : 0;
    for (int o = 16; o > 0; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if (lane == 0) s_w[w] = mine;
    __syncthreads();
    long long o = o0;
    for (int i = 0; i < w; ++i) o += s_w[i];
    const float4* __restrict__ src = e.xyzi + (size_t)b * e.max_points;
#pragma unroll 2
    for (int q = q0; q < q1; q += 32) {
        const int p = q + lane;
        const bool a = p < q1 && e.alive[base + p];
        float4 v;
        unsigned lab = 0;
        if (a) {
            if (p < s.n0) v = __ldg(&src[p]);
            else {
                const size_t t = (size_t)b * e.max_inserted + (p - s.n0);
                v = make_float4((float)e.tail_x[t], (float)e.tail_y[t], (float)e.tail_z[t], e.tail_i[t]);
            }
            lab = e.label[base + p];
            if constexpr (WORLD) world_point(wx, v.x, v.y, v.z);
        }
        const unsigned m = __ballot_sync(0xffffffffu, a);
        if (a) {
            const long long oo = o + __popc(m & ((1u << lane) - 1u));
            e.out_xyzi[oo] = v;
            e.out_label[oo] = lab;
        }
        o += __popc(m);
    }
}
