// Per-object point clouds built on the device from depth frames and instance-label images (DESIGN.md section 4.13).
//
// Stage A, gp_backproject_instances (one frame) and gp_backproject_frames (F frames of one size, objects numbered
// frame-major): back-projection and a stable segmented compaction, three launches.  The count and scatter grids are
// (tile groups of a frame, frame); one frame is the case F = 1 with objects [0, B) and the intrinsics as arguments.
//   count    one warp per tile of 1024 consecutive pixels (32 rounds of 32): per-tile object counts of the block's
//            frame into hist[object][tile of its frame] (__match_any_sync groups the lanes of one object, the lowest
//            lane adds the group); with F frames the block also clamps its frame's object range from frame_offsets
//   scan     one block per object: exclusive scan of its row of hist over the tiles, the row total into totals[object]
//   scatter  the count kernel's walk again: every block scans totals into the object offsets, a kept pixel lands at
//            offsets[object] + hist[object][tile] + (pixels of the object earlier in the tile) -- row-major pixel order
//            within each object, frames in order, whatever the scheduling, without atomics
#include <climits>
#include <cmath>

#include "common.cuh"
#include "philox.cuh"

namespace gp {
namespace clouds {

constexpr int WARPS = 4;        // warps (tiles) per block of the count and scatter kernels
constexpr int TILE = 1024;      // pixels per warp tile
constexpr int BATCH = 8;        // rounds loaded ahead of their processing
constexpr int SCAN_THREADS = 256;
constexpr int SAMPLE_THREADS = 256;

// exclusive scan of one int per thread over the block (blockDim.x a multiple of 32, <= 1024); total = block sum
__device__ __forceinline__ int block_exclusive_scan(int v, int &total) {
    __shared__ int warp_sums[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    int inc = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, d);
        if (lane >= d) inc += t;
    }
    if (lane == 31) warp_sums[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        int w = lane < nwarps ? warp_sums[lane] : 0;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, w, d);
            if (lane >= d) w += t;
        }
        warp_sums[lane] = w;   // inclusive
    }
    __syncthreads();
    total = warp_sums[nwarps - 1];
    const int before = warp == 0 ? 0 : warp_sums[warp - 1];
    __syncthreads();   // warp_sums may be reused by the caller's next scan
    return before + inc - v;
}

// object of pixel p (label b + 1 -> b) when the pixel is kept, else -1; n = objects of the pixel's frame
__device__ __forceinline__ int kept_object(int label, float z, int n) {
    return (label >= 1 && label <= n && z > 0.0f && isfinite(z)) ? label - 1 : -1;
}

// One stage-A call: F = gridDim.y frames of HW pixels, frame f at depth + f * HW.  frame_offsets == nullptr: one frame
// holding objects [0, B) (gp_backproject_instances); otherwise frame f holds the objects ranges[f] .. ranges[f+1]-1,
// which the count kernel derives from frame_offsets (clamp_range) and the scatter kernel reads back.
struct Frames {
    const float *depth;
    const int32_t *labels;
    int HW, B, n_tiles;               // n_tiles: tiles of one frame
    const float *intrinsics;          // [F][4] (fx, fy, cx, cy), or nullptr: the scatter kernel's arguments
    const int32_t *frame_offsets;     // [F+1] as given, or nullptr
    int *ranges;                      // [F+1] workspace: the clamped offsets
};

// The block's frame: its pixels and its objects lo .. lo + n - 1 (object label l of the frame is lo + l - 1).
struct FrameView {
    const float *depth;
    const int32_t *labels;
    int HW, n_tiles, lo, n;
};

__device__ __forceinline__ FrameView frame_view(const Frames &fr, int lo, int n) {
    const size_t first = (size_t)blockIdx.y * fr.HW;
    return FrameView{fr.depth + first, fr.labels + first, fr.HW, fr.n_tiles, lo, n};
}

// Frame f's object range [lo, hi) from frame_offsets, whatever it holds: offsets[0] is read as 0 and offsets[F] as B;
// in between offsets[g] is raised to the largest of offsets[1..g] and clamped into [0, B].  The ranges are then
// monotone, disjoint and cover [0, B), so every row of hist is written once and every output row is in bounds.
__device__ __forceinline__ void clamp_range(const Frames &fr, int f, int &lo, int &hi) {
    __shared__ int warp_max[WARPS];
    int m = INT_MIN;
    for (int g = 1 + threadIdx.x; g <= f; g += blockDim.x) m = max(m, __ldg(fr.frame_offsets + g));
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) warp_max[threadIdx.x >> 5] = m;
    __syncthreads();
#pragma unroll
    for (int w = 0; w < WARPS; ++w) m = max(m, warp_max[w]);
    lo = min(max(m, 0), fr.B);
    hi = f == (int)gridDim.y - 1 ? fr.B : max(lo, min(max(__ldg(fr.frame_offsets + f + 1), 0), fr.B));
}

// Walk warp `warp`'s tile of block blockIdx.x in pixel order, calling f(pixel, z, object, peers) once per round for
// every lane (object: frame-local, -1 for a dropped pixel or one past the frame); peers = the lanes of the round with
// the same object.
template <typename F>
__device__ __forceinline__ void walk_tile(const FrameView &fr, F &&f) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile = blockIdx.x * WARPS + warp;
    if (tile >= fr.n_tiles) return;
    const int base = tile * TILE;
    for (int r0 = 0; r0 < TILE / 32; r0 += BATCH) {
        int lab[BATCH];
        float z[BATCH];
#pragma unroll
        for (int i = 0; i < BATCH; ++i) {
            const int p = base + (r0 + i) * 32 + lane;
            lab[i] = p < fr.HW ? __ldg(fr.labels + p) : 0;
            z[i] = p < fr.HW ? __ldg(fr.depth + p) : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < BATCH; ++i) {
            const int obj = kept_object(lab[i], z[i], fr.n);
            const unsigned peers = __match_any_sync(0xffffffffu, obj);
            f(base + (r0 + i) * 32 + lane, z[i], obj, peers);
        }
        if (base + (r0 + BATCH) * 32 >= fr.HW) break;
    }
}

__global__ void __launch_bounds__(WARPS * 32) count_kernel(Frames frs, int *__restrict__ hist) {
    extern __shared__ int cnt[];   // [WARPS][n]
    int lo = 0, hi = frs.B;
    if (frs.frame_offsets) {
        clamp_range(frs, blockIdx.y, lo, hi);
        if (blockIdx.x == 0 && threadIdx.x == 0) {
            frs.ranges[blockIdx.y + 1] = hi;
            if (blockIdx.y == 0) frs.ranges[0] = 0;
        }
    }
    const FrameView fr = frame_view(frs, lo, hi - lo);
    for (int i = threadIdx.x; i < WARPS * fr.n; i += blockDim.x) cnt[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    int *mine = cnt + (threadIdx.x >> 5) * fr.n;
    walk_tile(fr, [&](int, float, int obj, unsigned peers) {
        if (obj >= 0 && lane == __ffs(peers) - 1) mine[obj] += __popc(peers);
        __syncwarp();
    });
    __syncthreads();
    // hist[obj][tile]: the WARPS tiles of a block are contiguous in each object's row
    const int tiles_here = min(WARPS, fr.n_tiles - (int)blockIdx.x * WARPS);
    for (int i = threadIdx.x; i < WARPS * fr.n; i += blockDim.x) {
        const int obj = i / WARPS, w = i % WARPS;
        if (w < tiles_here) hist[(size_t)(fr.lo + obj) * fr.n_tiles + blockIdx.x * WARPS + w] = cnt[w * fr.n + obj];
    }
}

__global__ void __launch_bounds__(SCAN_THREADS) scan_kernel(int *__restrict__ hist, int n_tiles, int *__restrict__ totals) {
    int *row = hist + (size_t)blockIdx.x * n_tiles;
    const int per = (n_tiles + SCAN_THREADS - 1) / SCAN_THREADS;
    const int lo = min(n_tiles, (int)threadIdx.x * per), hi = min(n_tiles, lo + per);
    int s = 0;
    for (int i = lo; i < hi; ++i) s += row[i];
    int total;
    int run = block_exclusive_scan(s, total);
    for (int i = lo; i < hi; ++i) {
        const int c = row[i];
        row[i] = run;
        run += c;
    }
    if (threadIdx.x == 0) totals[blockIdx.x] = total;
}

__global__ void __launch_bounds__(WARPS * 32) scatter_kernel(Frames frs, int W, float fx, float fy, float cx, float cy,
                                                             const int *__restrict__ hist,
                                                             const int *__restrict__ totals, float *__restrict__ xyz,
                                                             int32_t *__restrict__ offsets) {
    extern __shared__ int sm[];
    int *obj_off = sm;              // [B + 1]
    int *cnt = sm + frs.B + 1;      // [WARPS][n]: next output row of each object of the frame in each warp's tile
    const int B = frs.B;
    int lo = 0, n = B;
    if (frs.frame_offsets) {
        lo = frs.ranges[blockIdx.y];
        n = frs.ranges[blockIdx.y + 1] - lo;
        const float *in = frs.intrinsics + (size_t)blockIdx.y * 4;
        fx = in[0];
        fy = in[1];
        cx = in[2];
        cy = in[3];
    }
    const FrameView fr = frame_view(frs, lo, n);
    // object offsets = exclusive scan of totals (each block redoes this small scan: no fourth launch)
    const int per = (B + blockDim.x - 1) / blockDim.x;
    const int o_lo = min(B, (int)threadIdx.x * per), o_hi = min(B, o_lo + per);
    int s = 0;
    for (int i = o_lo; i < o_hi; ++i) s += totals[i];
    int total;
    int run = block_exclusive_scan(s, total);
    for (int i = o_lo; i < o_hi; ++i) {
        obj_off[i] = run;
        run += totals[i];
    }
    if (threadIdx.x == 0) obj_off[B] = total;
    __syncthreads();
    if (blockIdx.x == 0 && blockIdx.y == 0)
        for (int i = threadIdx.x; i <= B; i += blockDim.x) offsets[i] = obj_off[i];
    for (int i = threadIdx.x; i < WARPS * n; i += blockDim.x) {
        const int obj = i / WARPS, w = i % WARPS, tile = blockIdx.x * WARPS + w;
        if (tile < fr.n_tiles) cnt[w * n + obj] = obj_off[lo + obj] + hist[(size_t)(lo + obj) * fr.n_tiles + tile];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const unsigned lanes_below = (1u << lane) - 1u;
    int *mine = cnt + (threadIdx.x >> 5) * n;
    walk_tile(fr, [&](int p, float z, int obj, unsigned peers) {
        const int next = obj >= 0 ? mine[obj] : 0;
        __syncwarp();
        if (obj >= 0 && lane == __ffs(peers) - 1) mine[obj] = next + __popc(peers);
        __syncwarp();
        if (obj < 0) return;
        const int row = next + __popc(peers & lanes_below);
        const int v = p / W, u = p - v * W;
        // IEEE float32 in exactly this order: x = ((float)u - cx) * z / fx, y = ((float)v - cy) * z / fy
        float *o = xyz + (size_t)row * 3;
        o[0] = __fdiv_rn(__fmul_rn(__fsub_rn((float)u, cx), z), fx);
        o[1] = __fdiv_rn(__fmul_rn(__fsub_rn((float)v, cy), z), fy);
        o[2] = z;
    });
}

// pi_b: 4-round balanced Feistel network on k = max(2, ceil(log2 K)) bits (k rounded up to even), round function
// F_r(R) = Philox4x32-10(counter (R, r, 1, 0), key (lo32, hi32)).x & mask, cycle-walked into [0, K).
struct KeyedPermutation {
    uint32_t k0, k1, K, half, mask;

    __device__ KeyedPermutation(uint64_t key, uint32_t K_) : k0((uint32_t)key), k1((uint32_t)(key >> 32)), K(K_) {
        int k = K <= 1 ? 0 : 32 - __clz(K - 1);
        k = max(2, k);
        k += k & 1;
        half = (uint32_t)(k / 2);
        mask = (1u << half) - 1u;
    }
    __device__ __forceinline__ uint32_t encrypt(uint32_t x) const {
        uint32_t L = x >> half, R = x & mask;
#pragma unroll
        for (uint32_t r = 0; r < 4; ++r) {
            const uint32_t t = L ^ (philox4x32_10(make_uint4(R, r, 1u, 0u), k0, k1).x & mask);
            L = R;
            R = t;
        }
        return (L << half) | R;
    }
    __device__ __forceinline__ uint32_t operator()(uint32_t j) const {
        uint32_t y = encrypt(j);
        while (y >= K) y = encrypt(y);
        return y;
    }
};

__device__ __forceinline__ double block_sum(double v, double *red) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) v += __shfl_down_sync(0xffffffffu, v, d);
    if (lane == 0) red[warp] = v;
    __syncthreads();
    double s = 0.0;
    if (threadIdx.x == 0)
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += red[w];
    return s;   // thread 0 only
}

__global__ void __launch_bounds__(SAMPLE_THREADS) sample_kernel(const float *__restrict__ xyz, long long rows,
                                                                const int32_t *__restrict__ offsets,
                                                                const int64_t *__restrict__ keys, int N,
                                                                float *__restrict__ pts, float *__restrict__ center,
                                                                int32_t *__restrict__ counts) {
    __shared__ double red[3][SAMPLE_THREADS / 32];
    const int b = blockIdx.x;
    // offsets clamped into [0, rows]: malformed offsets give wrong clouds, never an out-of-bounds read
    const long long o0 = min(max((long long)offsets[b], 0ll), rows);
    const long long o1 = min(max((long long)offsets[b + 1], 0ll), rows);
    const uint32_t K = o1 > o0 ? (uint32_t)(o1 - o0) : 0u;
    float *out = pts + (size_t)b * N * 3;
    double sx = 0.0, sy = 0.0, sz = 0.0;
    if (K == 0) {
        for (size_t r = threadIdx.x; r < (size_t)N; r += blockDim.x) out[3 * r] = out[3 * r + 1] = out[3 * r + 2] = 0.0f;
    } else {
        const KeyedPermutation perm((uint64_t)keys[b], K);
        const uint32_t n = (uint32_t)N;
        const uint32_t tiled = K < n ? (n / K) * K : 0u;
        const float *src_base = xyz + (size_t)o0 * 3;
        for (size_t r = threadIdx.x; r < (size_t)N; r += blockDim.x) {   // size_t: 3 * r exceeds int for N > 2^31 / 3
            const uint32_t ur = (uint32_t)r;
            uint32_t src;
            if (K == n) src = ur;
            else if (ur < tiled) src = ur % K;                 // np.tile part
            else src = perm(K < n ? ur - tiled : ur);          // remainder / permutation(K)[:N]
            const float *p = src_base + (size_t)src * 3;
            const float x = p[0], y = p[1], z = p[2];
            out[3 * r] = x;
            out[3 * r + 1] = y;
            out[3 * r + 2] = z;
            sx += x;
            sy += y;
            sz += z;
        }
    }
    sx = block_sum(sx, red[0]);
    sy = block_sum(sy, red[1]);
    sz = block_sum(sz, red[2]);
    if (threadIdx.x == 0) {   // K == 0: every sum is 0.0, the centre is zeros
        center[3 * b] = (float)(sx / N);
        center[3 * b + 1] = (float)(sy / N);
        center[3 * b + 2] = (float)(sz / N);
        counts[b] = (int32_t)K;
    }
}

inline int n_tiles(int H, int W) { return (int)(((long long)H * W + TILE - 1) / TILE); }

// The three launches of stage A over F frames; the workspace holds hist [B][n_tiles], totals [B] and (F frames given
// by frame_offsets) the clamped offsets [F+1].
inline int launch_stage_a(const Frames &fr, int F, int W, float fx, float fy, float cx, float cy, float *xyz,
                          int32_t *offsets, int *hist, cudaStream_t st, const char *name) {
    int *totals = hist + (size_t)fr.B * fr.n_tiles;
    const dim3 grid((unsigned)((fr.n_tiles + WARPS - 1) / WARPS), (unsigned)F);
    count_kernel<<<grid, WARPS * 32, WARPS * fr.B * sizeof(int), st>>>(fr, hist);
    GP_CHECK_LAUNCH(name);
    scan_kernel<<<(unsigned)fr.B, SCAN_THREADS, 0, st>>>(hist, fr.n_tiles, totals);
    GP_CHECK_LAUNCH(name);
    scatter_kernel<<<grid, WARPS * 32, ((WARPS + 1) * fr.B + 1) * sizeof(int), st>>>(fr, W, fx, fy, cx, cy, hist,
                                                                                   totals, xyz, offsets);
    GP_CHECK_LAUNCH(name);
    return GP_OK;
}

}  // namespace clouds
}  // namespace gp

using namespace gp::clouds;

extern "C" size_t gp_backproject_instances_workspace_bytes(int H, int W, int B) {
    if (H < 1 || W < 1 || B < 1 || B > GP_MAX_FRAME_OBJECTS || (long long)H * W > GP_MAX_FRAME_PIXELS) return 0;
    return ((size_t)B * n_tiles(H, W) + (size_t)B) * sizeof(int);
}

extern "C" int gp_backproject_instances(const float *depth, const int32_t *labels, int H, int W, float fx, float fy,
                                        float cx, float cy, int B, float *xyz, int32_t *offsets, void *workspace,
                                        size_t workspace_bytes, gp_stream_t s) {
    GP_REQUIRE(H >= 1 && W >= 1 && B >= 1, "gp_backproject_instances: bad sizes H=%d W=%d B=%d", H, W, B);
    GP_REQUIRE((long long)H * W <= GP_MAX_FRAME_PIXELS, "gp_backproject_instances: frame %d x %d too large", H, W);
    if (B > GP_MAX_FRAME_OBJECTS) {
        gp::set_error("gp_backproject_instances: B=%d objects, at most %d supported", B, (int)GP_MAX_FRAME_OBJECTS);
        return GP_ERR_UNSUPPORTED;
    }
    GP_REQUIRE(depth && labels && xyz && offsets && workspace, "gp_backproject_instances: null pointer");
    GP_REQUIRE(std::isfinite(fx) && std::isfinite(fy) && std::isfinite(cx) && std::isfinite(cy) && fx != 0.0f &&
                   fy != 0.0f,
               "gp_backproject_instances: bad intrinsics fx=%g fy=%g cx=%g cy=%g", fx, fy, cx, cy);
    const size_t need = gp_backproject_instances_workspace_bytes(H, W, B);
    if (workspace_bytes < need) {
        gp::set_error("gp_backproject_instances: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return GP_ERR_WORKSPACE;
    }
    const Frames fr{depth, labels, H * W, B, n_tiles(H, W), nullptr, nullptr, nullptr};
    return launch_stage_a(fr, 1, W, fx, fy, cx, cy, xyz, offsets, (int *)workspace, gp::as_stream(s),
                          "gp_backproject_instances");
}

extern "C" size_t gp_backproject_frames_workspace_bytes(int F, int H, int W, int B) {
    if (F < 1 || F > GP_MAX_FRAMES || H < 1 || W < 1 || B < 1 || B > GP_MAX_FRAME_OBJECTS ||
        (long long)F * H * W > GP_MAX_FRAME_PIXELS)
        return 0;
    return ((size_t)B * n_tiles(H, W) + (size_t)B + (size_t)F + 1) * sizeof(int);
}

extern "C" int gp_backproject_frames(const float *depth, const int32_t *labels, int F, int H, int W,
                                     const float *intrinsics, const int32_t *frame_offsets, int B, float *xyz,
                                     int32_t *offsets, void *workspace, size_t workspace_bytes, gp_stream_t s) {
    GP_REQUIRE(F >= 1 && H >= 1 && W >= 1 && B >= 1, "gp_backproject_frames: bad sizes F=%d H=%d W=%d B=%d", F, H, W,
               B);
    GP_REQUIRE((long long)F * H * W <= GP_MAX_FRAME_PIXELS, "gp_backproject_frames: %d frames of %d x %d too large", F,
               H, W);
    if (B > GP_MAX_FRAME_OBJECTS || F > GP_MAX_FRAMES) {
        gp::set_error("gp_backproject_frames: F=%d frames and B=%d objects, at most %d and %d supported", F, B,
                      (int)GP_MAX_FRAMES, (int)GP_MAX_FRAME_OBJECTS);
        return GP_ERR_UNSUPPORTED;
    }
    GP_REQUIRE(depth && labels && intrinsics && frame_offsets && xyz && offsets && workspace,
               "gp_backproject_frames: null pointer");
    const size_t need = gp_backproject_frames_workspace_bytes(F, H, W, B);
    if (workspace_bytes < need) {
        gp::set_error("gp_backproject_frames: workspace of %zu bytes, %zu needed", workspace_bytes, need);
        return GP_ERR_WORKSPACE;
    }
    const int T = n_tiles(H, W);
    int *hist = (int *)workspace;
    int *ranges = hist + (size_t)B * T + B;
    const Frames fr{depth, labels, H * W, B, T, intrinsics, frame_offsets, ranges};
    return launch_stage_a(fr, F, W, 0.0f, 0.0f, 0.0f, 0.0f, xyz, offsets, hist, gp::as_stream(s),
                          "gp_backproject_frames");
}

extern "C" int gp_sample_points(const float *xyz, long long rows, const int32_t *offsets, const int64_t *keys, int B,
                                int N, float *pts, float *pts_center, int32_t *counts, gp_stream_t s) {
    GP_REQUIRE(B >= 1 && N >= 1 && rows >= 0, "gp_sample_points: bad sizes B=%d N=%d rows=%lld", B, N, rows);
    GP_REQUIRE(offsets && keys && pts && pts_center && counts && (xyz || rows == 0), "gp_sample_points: null pointer");
    sample_kernel<<<(unsigned)B, SAMPLE_THREADS, 0, gp::as_stream(s)>>>(xyz, rows, offsets, keys, N, pts, pts_center,
                                                                        counts);
    GP_CHECK_LAUNCH("gp_sample_points");
    return GP_OK;
}
