// ScoreNet / EnergyNet trunk kernels: weight packing, per-object head projection, single evaluation, energy
// scoring, the device-resident Dormand-Prince (scipy-RK45-faithful) integrator fused with the ScoreNet RHS (with
// scipy's dense output), and the fixed-step predictor-corrector sampler.  The MLP evaluation itself is a policy:
// SimtEval (FP32 FFMA, trunk.cuh), TcEval (tcgen05, 4-CTA clusters, trunk_tc.cuh), or TcSoloT / TcSolo (tcgen05, one
// CTA per tile, trunk_solo_t.cuh / trunk_solo.cuh); with_evaluator() picks one from an entry's `mode`.
#include <cuda_bf16.h>

#include <cstdlib>

#include "trunk_solo_t.cuh"

namespace gp {

// ------------------------------------------------------------------------------------------
// packing
// ------------------------------------------------------------------------------------------
struct RawTrunk {
    gp_trunk_params p;
};

// One 32-bit slot of a tensor-core weight image.  `row` holds k 0..nk-1 of the image's 64-wide k-atom (nk <= 64; k >= nk
// is zero), `which` the image of the pair, `wb` the slot's byte offset inside its 128-byte row and `logical16` its
// 16-byte unit with the SWIZZLE_128B XOR undone.
//   bf16 (TF32 = false): k = kl, kl + 1 of the atom as bf16 hi (which 0) or lo = bf16(w - hi) (which 1) parts;
//   tf32: k = 32 which + 4 logical16 + (wb % 16) / 4, rounded to tf32 (cvt.rna, the rounding of the A operand).
template <bool TF32>
__device__ __forceinline__ float pack_tc_slot(const float *row, size_t nk, size_t which, size_t logical16, size_t wb) {
    if (TF32) {
        const size_t k = 32 * which + logical16 * 4 + (wb % 16) / 4;
        return k < nk ? tc::tf32_rna(row[k]) : 0.f;
    }
    const size_t kl = logical16 * 8 + (wb % 16) / 2;    // k inside the 64-wide atom (even)
    float e[2];
    for (int t = 0; t < 2; ++t) {
        const float src = kl + t < nk ? row[kl + t] : 0.f;
        const float hi = __bfloat162float(__float2bfloat16_rn(src));
        e[t] = which == 0 ? hi : src - hi;
    }
    __nv_bfloat162 h2 = __floats2bfloat162_rn(e[0], e[1]);
    return *reinterpret_cast<float *>(&h2);
}

template <bool TF32>
__global__ void pack_trunk_kernel(RawTrunk raw, float *__restrict__ P) {
    const gp_trunk_params &p = raw.p;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < TrunkLayout::END; i += stride) {
        float v = 0.f;
        if (i < TrunkLayout::B1) {  // W1T[k][n] = pose_w0[n][k]
            const size_t k = i / 256, n = i % 256;
            v = p.pose_w0[n * 9 + k];
        } else if (i < TrunkLayout::W2T) {
            v = p.pose_b0[i - TrunkLayout::B1];
        } else if (i < TrunkLayout::B2) {  // W2T[k][n] = pose_w1[n][k]
            const size_t j = i - TrunkLayout::W2T, k = j / 256, n = j % 256;
            v = p.pose_w1[n * 256 + k];
        } else if (i < TrunkLayout::FOUR) {
            v = p.pose_b1[i - TrunkLayout::B2];
        } else if (i < TrunkLayout::WTT) {
            v = p.fourier_w[i - TrunkLayout::FOUR];
        } else if (i < TrunkLayout::BT) {  // WTT[k][j] = t_w[j][k]
            const size_t j = i - TrunkLayout::WTT, k = j / 128, n = j % 128;
            v = p.t_w[n * 128 + k];
        } else if (i < TrunkLayout::WHP) {
            v = p.t_b[i - TrunkLayout::BT];
        } else if (i < TrunkLayout::WHT) {  // WHP[h][k][j] = head_w0[h][j][1152+k]
            const size_t j = i - TrunkLayout::WHP, h = j / 65536, k = (j % 65536) / 256, n = j % 256;
            v = p.head_w0[h][n * 1408 + 1152 + k];
        } else if (i < TrunkLayout::WHF) {  // WHT[k][h*256+j] = head_w0[h][j][1024+k]
            const size_t j = i - TrunkLayout::WHT, k = j / 768, n = j % 768;
            v = p.head_w0[n / 256][(n % 256) * 1408 + 1024 + k];
        } else if (i < TrunkLayout::BH) {  // WHF[n][c] = head_w0[h][j][c]
            const size_t j = i - TrunkLayout::WHF, n = j / 1024, c = j % 1024;
            v = p.head_w0[n / 256][(n % 256) * 1408 + c];
        } else if (i < TrunkLayout::WO) {
            const size_t n = i - TrunkLayout::BH;
            v = p.head_b0[n / 256][n % 256];
        } else if (i < TrunkLayout::BO) {  // WO[n][o] = head_w1[h][o][j]
            const size_t j = i - TrunkLayout::WO, n = j / 4, o = j % 4;
            v = o < 3 ? p.head_w1[n / 256][o * 256 + (n % 256)] : 0.f;
        } else if (i < TrunkLayout::F32_END) {
            const size_t c = i - TrunkLayout::BO;
            v = c < 9 ? p.head_b1[c / 3][c % 3] : 0.f;
        } else if (i < TrunkLayout::W_TC) {
            v = 0.f;  // alignment padding
        } else if (i >= TrunkLayout::W_WIDE) {
            // wide head images of the cluster evaluator: [rank][kc][hi/lo] x [192 n][64 k]
            const size_t f = i - TrunkLayout::W_WIDE;
            const size_t per_img = TrunkLayout::WIDE_IMG_FLOATS;
            const size_t im = f / per_img, which = im % 2, kc = (im / 2) % 4, r = im / 8, o = (f % per_img) * 4;
            const size_t nl = o / 128, wb = o % 128;
            const size_t logical16 = (wb / 16) ^ (nl & 7);
            const size_t hh = nl / 64, n = 64 * r + nl % 64;
            v = pack_tc_slot<TF32>(p.head_w0[hh] + n * 1408 + 1152 + kc * 64, 64, which, logical16, wb);
        } else {
            // destination float slot -> (chunk q, image hi/lo, row n, 16-byte unit, element pair)
            const size_t f = i - TrunkLayout::W_TC;
            const size_t per_img = 128 * 64 / 2;
            // chunks 34..57 are the whole-head chunks of the one-CTA-per-tile evaluator (W_SOLO follows W_TC directly)
            const size_t q = f / (2 * per_img), which = (f / per_img) % 2, o = (f % per_img) * 4;
            const size_t nl = o / 128, wb = o % 128;
            const size_t logical16 = (wb / 16) ^ (nl & 7);      // undo the SWIZZLE_128B XOR
            const float *row;                                   // k 0.. of the image's k-atom
            size_t nk = 64;
            if (q < 2) {                 // pose_encoder.0: [256][9], zero-padded to k = 64
                row = p.pose_w0 + (q * 128 + nl) * 9;
                nk = 9;
            } else if (q < 10) {         // pose_encoder.2
                const size_t kc = (q - 2) / 2, nh = (q - 2) % 2, n = nh * 128 + nl;
                row = p.pose_w1 + n * 256 + kc * 64;
            } else if (q < TrunkLayout::TC_CHUNKS) {   // head columns of one cluster rank, two k-atoms per image
                const size_t r = (q - 10) / 6, hh = ((q - 10) % 6) / 2, j = (q - 10) % 2;
                const size_t kc = 2 * j + nl / 64, n = 64 * r + nl % 64;
                row = p.head_w0[hh] + n * 1408 + 1152 + kc * 64;
            } else {                     // whole heads: [h][kc][nh] images of [128 n][64 k]
                const size_t qs = q - TrunkLayout::TC_CHUNKS;
                const size_t hh = qs / 8, kc = (qs % 8) / 2, nh = qs % 2, n = nh * 128 + nl;
                row = p.head_w0[hh] + n * 1408 + 1152 + kc * 64;
            }
            v = pack_tc_slot<TF32>(row, nk, which, logical16, wb);
        }
        P[i] = v;
    }
}

// ------------------------------------------------------------------------------------------
// per-object projection  proj[b][n] = bh[n] + sum_c WHF[n][c] * pts_feat[b][c]
// block: 8 warps; 8 objects x 64 outputs per block; one warp per output, lanes stride c.
// ------------------------------------------------------------------------------------------
constexpr int PJ_OBJ = 8, PJ_OUT = 64;
__global__ void __launch_bounds__(256)
project_kernel(const float *__restrict__ P, const float *__restrict__ feat, int B, float *__restrict__ proj) {
    __shared__ __align__(16) float s_f[PJ_OBJ][1024];
    const int b0 = blockIdx.y * PJ_OBJ, n0 = blockIdx.x * PJ_OUT;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < PJ_OBJ * 256; i += 256) {
        const int o = i >> 8, c4 = i & 255;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (b0 + o < B) v = __ldg(reinterpret_cast<const float4 *>(feat + (size_t)(b0 + o) * 1024) + c4);
        reinterpret_cast<float4 *>(&s_f[o][0])[c4] = v;
    }
    __syncthreads();
    // a warp takes two outputs at a time and requests both weight rows (2 x 8 16-byte loads per lane) before the first FMA:
    // 4 L2 round trips per warp instead of 32 (the launch sits between the encoder and the sampler: latency is what counts)
    for (int j = 2 * warp; j < PJ_OUT; j += 16) {
        float4 wv[2][8];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const float4 *w = reinterpret_cast<const float4 *>(P + TrunkLayout::WHF + (size_t)(n0 + j + u) * 1024);
#pragma unroll
            for (int i = 0; i < 8; ++i) wv[u][i] = __ldg(w + lane + 32 * i);
        }
        float acc[2][PJ_OBJ];
#pragma unroll
        for (int u = 0; u < 2; ++u)
#pragma unroll
            for (int o = 0; o < PJ_OBJ; ++o) acc[u][o] = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
#pragma unroll
            for (int o = 0; o < PJ_OBJ; ++o) {
                const float4 f = reinterpret_cast<const float4 *>(&s_f[o][0])[lane + 32 * i];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    acc[u][o] = fmaf(f.x, wv[u][i].x, acc[u][o]);
                    acc[u][o] = fmaf(f.y, wv[u][i].y, acc[u][o]);
                    acc[u][o] = fmaf(f.z, wv[u][i].z, acc[u][o]);
                    acc[u][o] = fmaf(f.w, wv[u][i].w, acc[u][o]);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int n = n0 + j + u;
            const float bias = __ldg(P + TrunkLayout::BH + n);
#pragma unroll
            for (int o = 0; o < PJ_OBJ; ++o) {
                float v = acc[u][o];
#pragma unroll
                for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
                if (lane == 0 && b0 + o < B) proj[(size_t)(b0 + o) * 768 + n] = v + bias;
            }
        }
    }
}

// ------------------------------------------------------------------------------------------
// Evaluator policies: how one tile of rows gets its f_theta.  Every kernel below is a template over one of them, and
// they all expose the same shared-memory members (x, out, obj, tq, four, tfeat, times, red) to the integrator code.
//   SimtEval<RPT>    FP32 FFMA, 4*RPT rows, 256 threads, one CTA per tile (trunk.cuh)
//   TcEval<NPASS>    tcgen05, 128 rows, 320 threads, a 4-CTA cluster per tile (trunk_tc.cuh)
//   TcSoloT<NPASS>   tcgen05, 128 rows, 320 threads, one CTA per tile, A operand in tensor memory (trunk_solo_t.cuh)
//   TcSolo<NPASS>    the same with the A operand in shared memory (trunk_solo.cuh)
// NPASS is the number of MMAs per product: 1 bf16, 2 tf32, 3 split-bf16.  with_evaluator() picks one for an entry.
// ------------------------------------------------------------------------------------------
// Tile loop of the evaluators without a cluster: CTA b takes tiles b, b + gridDim.x, ... and stores its own results.
struct OneCtaPerTile {
    static constexpr int CLUSTER = 1;     // CTAs that share a tile
    static __device__ __forceinline__ int tile_first() { return blockIdx.x; }
    static __device__ __forceinline__ int tile_step() { return gridDim.x; }
    template <class Ctx>
    static __device__ __forceinline__ bool writer(const Ctx &) { return true; }
    template <class Ctx>
    static __device__ __forceinline__ size_t replica_index(const Ctx &) { return 0; }
    static __device__ __forceinline__ void tile_sync() {}
};

template <int RPT>
struct SimtEval : OneCtaPerTile {
    static constexpr int RT = 4 * RPT;
    static constexpr int NT = SIMT_THREADS;
    static constexpr int XS = 12;         // row stride of the input / output tile
    static constexpr int TQW = 768;       // t-branch columns held per stage
    using Smem = TileSmem<RPT>;
    using Ctx = SimtCtx;
    static constexpr size_t smem_bytes() { return sizeof(Smem) + 16; }
    static __device__ __forceinline__ Smem &smem(unsigned char *raw) {
        // pointer arithmetic on the __shared__ array keeps the shared address space (LDS/STS, not generic LD/ST)
        return *reinterpret_cast<Smem *>(raw + ((16u - (tc::smem_u32(raw) & 15u)) & 15u));
    }
    static __device__ __forceinline__ float *xin(Smem &S) { return S.x; }
    static __device__ __forceinline__ float *outp(Smem &S) { return S.out[0]; }
    static __device__ __forceinline__ float *tq(Smem &S) { return S.tq; }
    static __device__ __forceinline__ void setup(Smem &S, Ctx &c, const float *P) { simt_setup(S, c, P); }
    static __device__ __forceinline__ void teardown(Smem &S, Ctx &c) { simt_teardown(S, c); }
    // t-branch of the ns stage times in S.times -> S.tq[ns][TQW]
    static __device__ __forceinline__ void stage_tq(const float *P, Smem &S, Ctx &, int ns) {
        compute_tq(P, S.times, ns, S.tqs, S.tq);
    }
    static __device__ __forceinline__ void begin_tile(Smem &S, Ctx &, const float *, int r0, int N, int rpo) {
        for (int r = threadIdx.x; r < RT; r += NT) S.obj[r] = (r0 + r < N) ? (r0 + r) / rpo : -1;
    }
    static __device__ __forceinline__ void forward(const float *P, const float *proj, Smem &S, Ctx &c, const float *tq) {
        tile_forward<RPT>(P, proj, S, c, tq);
    }
    static __device__ __forceinline__ void report(Ctx &, double *) {}
};

template <int NPASS>
struct TcEval {
    static constexpr int RT = tc::RT;
    static constexpr int NT = tc::NTHREADS;
    static constexpr int XS = tc::XS;
    static constexpr int TQW = tc::NHC;   // only the head columns this cluster rank owns
    static constexpr int CLUSTER = tc::CL;
    using Smem = tc::Smem<NPASS>;
    using Ctx = tc::State;
    static constexpr size_t smem_bytes() { return sizeof(Smem) + 1024; }
    static __device__ __forceinline__ Smem &smem(unsigned char *raw) {
        return *reinterpret_cast<Smem *>(((uintptr_t)raw + 1023) & ~(uintptr_t)1023);
    }
    // the CTAs of a cluster work on the same tile and run the code around forward() replicated
    static __device__ __forceinline__ int tile_first() { return (int)tc::cluster_id_x(); }
    static __device__ __forceinline__ int tile_step() { return (int)tc::cluster_count_x(); }
    static __device__ __forceinline__ bool writer(const Ctx &c) { return c.rank == 0; }
    static __device__ __forceinline__ size_t replica_index(const Ctx &c) { return c.rank; }
    static __device__ __forceinline__ void tile_sync() { tc::cluster_arrive(); tc::cluster_wait(); }
    static __device__ __forceinline__ float *xin(Smem &S) { return S.x; }
    static __device__ __forceinline__ float *outp(Smem &S) { return S.x; }   // forward() overwrites its inputs
    static __device__ __forceinline__ float *tq(Smem &S) { return S.tq; }
    static __device__ __forceinline__ void setup(Smem &S, Ctx &c, const float *P) { tc::setup<NPASS>(S, c, P); }
    static __device__ __forceinline__ void teardown(Smem &S, Ctx &c) { tc::teardown<NPASS>(S, c); }
    static __device__ __forceinline__ void stage_tq(const float *P, Smem &S, Ctx &c, int ns) { tc::compute_tq_rank<NPASS>(P, S, c, ns); }
    static __device__ __forceinline__ void begin_tile(Smem &S, Ctx &c, const float *proj, int r0, int N, int rpo) {
        tc::begin_tile<NPASS>(S, c, proj, r0, N, rpo);
    }
    static __device__ __forceinline__ void forward(const float *P, const float *proj, Smem &S, Ctx &c, const float *tq) {
        tc::forward<NPASS>(P, proj, S, c, tq);
    }
    // phase cycle counters of epilogue thread 0 of CTA 0 (profiling aid, stats[8..13]; stats[14] = whole kernel)
    static __device__ __forceinline__ void report(Ctx &c, double *stats) {
        if (blockIdx.x == 0 && threadIdx.x == 64) {
            stats[8] = (double)c.cyc_fwd; stats[9] = (double)c.cyc_l1; stats[10] = (double)c.cyc_wait1;
            stats[11] = (double)c.cyc_epi1; stats[12] = (double)c.cyc_waith; stats[13] = (double)c.cyc_epi2;
            for (int i = 0; i < 5; ++i) stats[20 + i] = (double)c.cyc_x[i];
        }
        if (blockIdx.x == 0 && threadIdx.x == 32) stats[15] = (double)c.cyc_wfull;   // the MMA issuer's own counter
    }
};

// One CTA per 128-row tile, no cluster: the throughput shape for batches of more tiles than the GPU has clusters.
// One copy of the integrator state.  TcSoloT and TcSolo share everything here and differ in where A lives.
template <class SmemT, class CtxT>
struct TcSoloTile : OneCtaPerTile {
    static constexpr int RT = tc::RT;
    static constexpr int NT = tc::NTHREADS;
    static constexpr int XS = tc::XS;
    static constexpr int TQW = 768;
    using Smem = SmemT;
    using Ctx = CtxT;
    static constexpr size_t smem_bytes() { return sizeof(Smem) + 1024; }
    static __device__ __forceinline__ Smem &smem(unsigned char *raw) {
        return *reinterpret_cast<Smem *>(((uintptr_t)raw + 1023) & ~(uintptr_t)1023);
    }
    static __device__ __forceinline__ float *xin(Smem &S) { return S.x; }
    static __device__ __forceinline__ float *outp(Smem &S) { return S.x; }   // forward() overwrites its inputs
    static __device__ __forceinline__ float *tq(Smem &S) { return S.tq; }
    static __device__ __forceinline__ void report(Ctx &c, double *stats) {
        if (blockIdx.x == 0 && threadIdx.x == 64) {
            stats[8] = (double)c.cyc_fwd; stats[9] = (double)c.cyc_l1; stats[10] = (double)c.cyc_wait1;
            stats[11] = (double)c.cyc_epi1; stats[12] = (double)c.cyc_waith; stats[13] = (double)c.cyc_epi2;
            stats[20] = (double)c.cyc_tail;
        }
    }
};
// A operand in tensor memory (trunk_solo_t.cuh).
template <int NPASS>
struct TcSoloT : TcSoloTile<solot::Smem<NPASS>, solot::State> {
    using Smem = solot::Smem<NPASS>;
    using Ctx = solot::State;
    static __device__ __forceinline__ void setup(Smem &S, Ctx &c, const float *P) { solot::setup<NPASS>(S, c, P); }
    static __device__ __forceinline__ void teardown(Smem &S, Ctx &c) { solot::teardown<NPASS>(S, c); }
    static __device__ __forceinline__ void stage_tq(const float *P, Smem &S, Ctx &, int ns) { solot::compute_tq_all<NPASS>(P, S, ns); }
    static __device__ __forceinline__ void begin_tile(Smem &S, Ctx &c, const float *proj, int r0, int N, int rpo) {
        solot::begin_tile<NPASS>(S, c, proj, r0, N, rpo);
    }
    static __device__ __forceinline__ void forward(const float *P, const float *proj, Smem &S, Ctx &c, const float *tq) {
        solot::forward<NPASS>(P, proj, S, c, tq);
    }
};
// A operand in shared memory (trunk_solo.cuh).
template <int NPASS>
struct TcSolo : TcSoloTile<solo::Smem<NPASS>, solo::State> {
    using Smem = solo::Smem<NPASS>;
    using Ctx = solo::State;
    static __device__ __forceinline__ void setup(Smem &S, Ctx &c, const float *P) { solo::setup<NPASS>(S, c, P); }
    static __device__ __forceinline__ void teardown(Smem &S, Ctx &c) { solo::teardown<NPASS>(S, c); }
    static __device__ __forceinline__ void stage_tq(const float *P, Smem &S, Ctx &, int ns) { solo::compute_tq_all<NPASS>(P, S, ns); }
    static __device__ __forceinline__ void begin_tile(Smem &S, Ctx &c, const float *proj, int r0, int N, int rpo) {
        solo::begin_tile<NPASS>(S, c, proj, r0, N, rpo);
    }
    static __device__ __forceinline__ void forward(const float *P, const float *proj, Smem &S, Ctx &c, const float *tq) {
        solo::forward<NPASS>(P, proj, S, c, tq);
    }
};

// Each evaluator's dynamic shared memory leaves room for the static shared memory of the kernels built on it (stage
// constants, per-row t) in the 227 KB of a CTA.
template <class... EV>
constexpr bool smem_fits() { return ((EV::smem_bytes() + 768 <= 227 * 1024) && ...); }
static_assert(smem_fits<SimtEval<2>, SimtEval<4>, SimtEval<6>, SimtEval<8>, TcEval<1>, TcEval<2>, TcEval<3>, TcSoloT<1>,
                        TcSoloT<2>, TcSoloT<3>, TcSolo<1>, TcSolo<3>>(),
              "evaluator shared memory exceeds 227 KB");
static_assert(sizeof(solot::Smem<2>) == sizeof(solot::Smem<3>) && sizeof(tc::Smem<2>) == sizeof(tc::Smem<3>),
              "tf32 mode uses the split mode's ring");

// ------------------------------------------------------------------------------------------
// single evaluation / energy: one CTA per tile; rows may carry different t (handled by runs)
// MODE 0: score = f/(std+1e-7) -> out [N,9];  MODE 1: energy [N,2] from f64 poses
// ------------------------------------------------------------------------------------------
struct EvalArgs {
    const float *P, *proj, *x;
    const double *poses;
    const float *center, *t;
    int N, rpo;
    float *out;
};

template <class EV, int MODE>
__global__ void __launch_bounds__(EV::NT, 1) eval_kernel(EvalArgs a) {
    const float *__restrict__ P = a.P, *__restrict__ proj = a.proj, *__restrict__ x = a.x;
    const double *__restrict__ poses = a.poses;
    const float *__restrict__ center = a.center, *__restrict__ t = a.t;
    const int N = a.N, rpo = a.rpo;
    float *__restrict__ out = a.out;
    constexpr int RT = EV::RT, NT = EV::NT, XS = EV::XS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typename EV::Smem &S = EV::smem(smem_raw);
    typename EV::Ctx ctx;
    const int tid = threadIdx.x;
    const int r0 = EV::tile_first() * RT;
    EV::setup(S, ctx, P);
    __shared__ float s_trow[EV::RT];
    EV::begin_tile(S, ctx, proj, r0, N, rpo);
    for (int r = tid; r < RT; r += NT) s_trow[r] = (r0 + r < N) ? t[r0 + r] : 0.f;
    __syncthreads();
    const int nrows = min(RT, N - r0);
    int run0 = 0;
    while (run0 < nrows) {  // maximal runs of equal t share one t-branch evaluation
        const float tv = s_trow[run0];
        int run1 = run0 + 1;
        while (run1 < nrows && s_trow[run1] == tv) ++run1;
        // (re)load the inputs: the evaluator may reuse the input buffer for its outputs
        float *xin = EV::xin(S);
        for (int i = tid; i < RT * XS; i += NT) {
            const int r = i / XS, c = i - XS * r;
            float v = 0.f;
            if (r0 + r < N && c < 9) {
                if (MODE == 0) {
                    v = x[(size_t)(r0 + r) * 9 + c];
                } else {
                    // pose_samples.type_as(f32) then [:, -3:] -= pts_center (posenet_agent.py:668-694)
                    v = (float)poses[(size_t)(r0 + r) * 9 + c];
                    if (c >= 6) v = v - center[(size_t)(r0 + r) * 3 + (c - 6)];
                }
            }
            xin[i] = v;
        }
        if (tid == 0) S.times[0] = tv;
        __syncthreads();
        float xr[9];  // this thread's row for the energy inner products (kept across the evaluation)
        if (MODE == 1) {
#pragma unroll
            for (int c = 0; c < 9; ++c) xr[c] = (run0 + tid < run1) ? xin[(run0 + tid) * XS + c] : 0.f;
        }
        EV::stage_tq(P, S, ctx, 1);
        EV::forward(P, proj, S, ctx, EV::tq(S));
        const float *fo = EV::outp(S);
        const float std = sigma_f32(tv);
        if (!EV::writer(ctx)) {
            // replicated CTAs of a cluster hold the same result; one of them stores it
        } else if (MODE == 0) {
            for (int i = tid; i < (run1 - run0) * 9; i += NT) {
                const int r = run0 + i / 9, c = i % 9;
                out[(size_t)(r0 + r) * 9 + c] = fo[r * XS + c] / (std + 1e-7f);
            }
        } else {
            static_assert(EV::RT <= EV::NT, "one thread per row");
            const int r = run0 + tid;
            if (r < run1) {
                float er = 0.f, et = 0.f;
#pragma unroll
                for (int c = 0; c < 6; ++c) er += xr[c] * (fo[r * XS + c] / std);
#pragma unroll
                for (int c = 6; c < 9; ++c) et += xr[c] * (fo[r * XS + c] / std);
                out[(size_t)(r0 + r) * 2 + 0] = er;
                out[(size_t)(r0 + r) * 2 + 1] = et;
            }
        }
        __syncthreads();
        run0 = run1;
    }
    EV::teardown(S, ctx);
}

// ------------------------------------------------------------------------------------------
// Dormand-Prince 5(4) with scipy's controller, device resident.
// ------------------------------------------------------------------------------------------
__constant__ double c_C[6] = {0.0, 1.0 / 5, 3.0 / 10, 4.0 / 5, 8.0 / 9, 1.0};
__constant__ double c_A[6][5] = {
    {0, 0, 0, 0, 0},
    {1.0 / 5, 0, 0, 0, 0},
    {3.0 / 40, 9.0 / 40, 0, 0, 0},
    {44.0 / 45, -56.0 / 15, 32.0 / 9, 0, 0},
    {19372.0 / 6561, -25360.0 / 2187, 64448.0 / 6561, -212.0 / 729, 0},
    {9017.0 / 3168, -355.0 / 33, 46732.0 / 5247, 49.0 / 176, -5103.0 / 18656}};
__constant__ double c_B[6] = {35.0 / 384, 0, 500.0 / 1113, 125.0 / 192, -2187.0 / 6784, 11.0 / 84};
__constant__ double c_E[7] = {-71.0 / 57600, 0, 71.0 / 16695, -71.0 / 1920, 17253.0 / 339200, -22.0 / 525, 1.0 / 40};

// dense-output coefficients (scipy rk.py RK45.P, [7 stages][4 powers])
__constant__ double c_P[7][4] = {
    {1.0, -8048581381.0 / 2820520608.0, 8663915743.0 / 2820520608.0, -12715105075.0 / 11282082432.0},
    {0.0, 0.0, 0.0, 0.0},
    {0.0, 131558114200.0 / 32700410799.0, -68118460800.0 / 10900136933.0, 87487479700.0 / 32700410799.0},
    {0.0, -1754552775.0 / 470086768.0, 14199869525.0 / 1410260304.0, -10690763975.0 / 1880347072.0},
    {0.0, 127303824393.0 / 49829197408.0, -318862633887.0 / 49829197408.0, 701980252875.0 / 199316789632.0},
    {0.0, -282668133.0 / 205662961.0, 2019193451.0 / 616988883.0, -1453857185.0 / 822651844.0},
    {0.0, 40617522.0 / 29380423.0, -110615467.0 / 29380423.0, 69997945.0 / 29380423.0}};

struct OdeArgs {
    const float *P;
    const float *proj;
    const double *x0;
    const float *center;
    int N, rpo;
    double T, eps, rtol, atol;
    int denoise;
    double denoise_steps;   // the denoise step is (1 - eps) / denoise_steps (1000, or num_steps with dense output)
    const double *t_eval;   // dense output: n_eval times in integration order (device), or nullptr
    int n_eval;
    double *dense;          // [n_eval][N][9] raw states at t_eval
    double *x_out;
    double *traj;
    int max_traj;
    double *stats;
    // workspace
    double *y[2];     // current / candidate state   [N][9]
    double *K[7];     // stage derivatives K[0..6]    [N][9]
    size_t replica;   // doubles between the private copies of y / K of the CTAs that share a tile (cluster evaluator)
    double *part;     // [2][3][ntiles] partial sums
    unsigned int *gbar;  // grid barrier counter (zeroed before the launch)
    int ntiles;
};

// Grid-wide barrier of a launch whose CTAs are all resident (cooperative launch): one arrival per CTA on a
// monotonically increasing counter (zeroed by the host before the launch), thread 0 spins on an acquire load.
// `target` is this thread's running count of expected arrivals.
__device__ __forceinline__ void grid_barrier(unsigned int *counter, unsigned int &target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        target += gridDim.x;
        __threadfence();  // release: the CTA's global writes (made visible to thread 0 by the barrier above) first
        atomicAdd(counter, 1u);
        unsigned int v;
        do {
            asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(counter) : "memory");
        } while (v < target);
    }
    __syncthreads();
}

// sum part[0..ntiles) in a fixed order; identical in every CTA
__device__ __forceinline__ double grid_total(const double *part, int ntiles, double *s_red) {
    double v = 0.0;
    for (int i = threadIdx.x; i < ntiles; i += blockDim.x) v += __ldcg(part + i);
    return block_sum(v, s_red);
}

// The pieces of a Runge-Kutta step that touch the float64 state.  They are separate (not inlined) functions:
// each gets its own register allocation (the integrator around them keeps ~100 live values) and the kernel's
// code stays small -- it runs once per step, so instruction fetch matters.
// inputs of stage S (1..5: y + h * sum_j a_Sj K_j; 6: y_new, also stored) for one tile -> xin (float32).
// All loads of a thread are issued before any use: one memory round trip per stage.
// 4 consecutive float64 values (32-byte aligned)
struct D4 { double v[4]; };
__device__ __forceinline__ D4 ld_d4(const double *p) {
    const double2 a = *reinterpret_cast<const double2 *>(p), b = *reinterpret_cast<const double2 *>(p + 2);
    return D4{{a.x, a.y, b.x, b.y}};
}

// inputs of stage S (1..5: y + h * sum_j a_Sj K_j; 6: y_new, also stored) for one tile -> xin (float32).
// Thread t owns elements 4t..4t+3 of the tile; its loads are unconditional (the buffers are padded to whole
// tiles) and all issued before the first use: one memory round trip per stage.
// this thread's quad of scipy's `fun` from the evaluator's output tile: K = 0 - coef * f_theta / (std + 1e-7)
// (scorenet.py:262-264, samplers.py:219)
template <class EV>
__device__ __forceinline__ D4 rhs_quad(const float *fo, int q, float std, double coef) {
    constexpr int XS = EV::XS;
    float f[4];
    if (XS == 9) {
        const float4 v = *reinterpret_cast<const float4 *>(fo + 4 * q);
        f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
    } else {
#pragma unroll
        for (int e = 0; e < 4; ++e) f[e] = fo[((4 * q + e) / 9) * XS + (4 * q + e) % 9];
    }
    D4 k;
#pragma unroll
    for (int e = 0; e < 4; ++e) k.v[e] = 0.0 - coef * (double)(f[e] / (std + 1e-7f));
    return k;
}
__device__ __forceinline__ void st_d4(double *p, const D4 &v) {
    *reinterpret_cast<double2 *>(p) = make_double2(v.v[0], v.v[1]);
    *reinterpret_cast<double2 *>(p + 2) = make_double2(v.v[2], v.v[3]);
}

// `k_store` (stages 2..6): the derivative of the previous stage has not been written yet -- it is formed here from the
// evaluator's output tile `fo` (which the same thread then overwrites with the new inputs when the evaluator reuses
// its input buffer), stored to k_store and used from registers: no separate pass over the tile, no extra barrier.
template <class EV, int S>
__device__ __noinline__ void ode_stage_input(const double *y, double *ynew, const double *k0, const double *k1,
                                             const double *k2, const double *k3, const double *k4, const double *k5,
                                             float *xin, int tile, int N, double h, const float *fo, double *k_store,
                                             float std_prev, double coef_prev) {
    constexpr int RT = EV::RT, XS = EV::XS;
    constexpr int NK = S < 6 ? S : 6;
    static_assert(RT * 9 / 4 <= EV::NT && (RT * 9) % 4 == 0, "one quad per thread");
    const int q = threadIdx.x;
    if (q < RT * 9 / 4) {
        const size_t g = (size_t)tile * RT * 9 + 4 * q;
        const int nvalid = min(RT, N - tile * RT) * 9;
        const double *const ks[6] = {k0, k1, k2, k3, k4, k5};
        D4 kv[NK];
        const D4 yv = ld_d4(y + g);
#pragma unroll
        for (int j = 0; j < NK; ++j)
            if (!(k_store != nullptr && j == S - 1)) kv[j] = ld_d4(ks[j] + g);
        if (k_store != nullptr) {
            kv[S - 1 < NK ? S - 1 : NK - 1] = rhs_quad<EV>(fo, q, std_prev, coef_prev);
            st_d4(k_store + g, kv[S - 1 < NK ? S - 1 : NK - 1]);
        }
        float v[4];
        D4 yn;
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            double acc = 0.0;
            if (S < 6) {
#pragma unroll
                for (int j = 0; j < NK; ++j) acc += kv[j].v[e] * c_A[S][j];
                yn.v[e] = yv.v[e] + acc * h;  // dy = dot(K[:s].T, a[:s]) * h
            } else {
#pragma unroll
                for (int j = 0; j < 6; ++j) acc += kv[j].v[e] * c_B[j];
                yn.v[e] = yv.v[e] + h * acc;  // y_new = y + h * dot(K[:-1].T, B)
            }
            v[e] = 4 * q + e < nvalid ? (float)yn.v[e] : 0.f;
        }
        if (S == 6) {
            *reinterpret_cast<double2 *>(ynew + g) = make_double2(yn.v[0], yn.v[1]);
            *reinterpret_cast<double2 *>(ynew + g + 2) = make_double2(yn.v[2], yn.v[3]);
        }
        if (XS == 9) {
            *reinterpret_cast<float4 *>(xin + 4 * q) = make_float4(v[0], v[1], v[2], v[3]);
        } else {
#pragma unroll
            for (int e = 0; e < 4; ++e) xin[((4 * q + e) / 9) * XS + (4 * q + e) % 9] = v[e];  // padding columns stay zero
        }
    }
    __syncthreads();
}

// K_dst = -0.5 g(t)^2 * score for one tile (scipy's `fun`): score = f_theta / (std + 1e-7) (scorenet.py:262-264),
// samplers.py:219
template <class EV>
__device__ __noinline__ void ode_store_k(const float *fo, double *Kd, int tile, int N, float std, double coef) {
    constexpr int RT = EV::RT, NT = EV::NT, XS = EV::XS;
    const int r0 = tile * RT;
    for (int i = threadIdx.x; i < RT * 9; i += NT) {
        const int r = i / 9, c = i - 9 * r;
        if (r0 + r < N) {
            const float sc = fo[r * XS + c] / (std + 1e-7f);
            Kd[(size_t)(r0 + r) * 9 + c] = 0.0 - coef * (double)sc;
        }
    }
    __syncthreads();
}

// this thread's share of sum((h * K^T E / scale)^2) over one tile (rk.py:139-147); candidate state -> traj_slot
template <class EV>
__device__ __noinline__ double ode_error_part(const double *y, const double *ynew, const double *k0, const double *k1,
                                              const double *k2, const double *k3, const double *k4, const double *k5,
                                              double *k6, int tile, int N, double h, double atol, double rtol,
                                              double *traj_slot, const float *fo, float std6, double coef6) {
    constexpr int RT = EV::RT;
    const int q = threadIdx.x;
    double se = 0.0;
    if (q < RT * 9 / 4) {
        const size_t g = (size_t)tile * RT * 9 + 4 * q;
        const int nvalid = min(RT, N - tile * RT) * 9;
        const double *const ks[6] = {k0, k1, k2, k3, k4, k5};
        D4 kv[7];
        const D4 y0 = ld_d4(y + g), y1 = ld_d4(ynew + g);
#pragma unroll
        for (int j = 0; j < 6; ++j) kv[j] = ld_d4(ks[j] + g);
        kv[6] = rhs_quad<EV>(fo, q, std6, coef6);   // f(t + h, y_new): formed from the evaluator's output, kept for FSAL
        st_d4(k6 + g, kv[6]);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            double ev = 0.0;
#pragma unroll
            for (int j = 0; j < 7; ++j) ev += kv[j].v[e] * c_E[j];
            ev *= h;
            const double sc = atol + fmax(fabs(y0.v[e]), fabs(y1.v[e])) * rtol;
            if (4 * q + e < nvalid) {
                se += (ev / sc) * (ev / sc);
                if (traj_slot) traj_slot[g + e] = y1.v[e];  // speculative: kept only if the step is accepted
            }
        }
    }
    return se;
}

// Dense output of an accepted step (scipy rk.py:715-737, RkDenseOutput): y(te) = y_old + h * Q . [x, x^2, x^3, x^4],
// Q = K^T . P, x = (te - t_old) / h, for the quads of one tile -> dst (the tile's first row).
template <class EV>
__device__ __noinline__ void ode_dense_point(const double *y, const double *k0, const double *k1, const double *k2,
                                             const double *k3, const double *k4, const double *k5, const double *k6,
                                             int tile, int N, double h, double x, double *dst) {
    constexpr int RT = EV::RT;
    const int q = threadIdx.x;
    if (q >= RT * 9 / 4) return;
    const size_t g = (size_t)tile * RT * 9 + 4 * q;
    const int nvalid = min(RT, N - tile * RT) * 9;
    const double *const ks[7] = {k0, k1, k2, k3, k4, k5, k6};
    const double p1 = x, p2 = p1 * x, p3 = p2 * x, p4 = p3 * x;   // np.cumprod([x, x, x, x])
    const D4 yv = ld_d4(y + g);
    D4 kv[7];
#pragma unroll
    for (int j = 0; j < 7; ++j) kv[j] = ld_d4(ks[j] + g);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        double qc[4] = {0.0, 0.0, 0.0, 0.0};
#pragma unroll
        for (int j = 0; j < 7; ++j)
#pragma unroll
            for (int c = 0; c < 4; ++c) qc[c] += kv[j].v[e] * c_P[j][c];
        const double v = yv.v[e] + h * (((qc[0] * p1 + qc[1] * p2) + qc[2] * p3) + qc[3] * p4);
        if (4 * q + e < nvalid) dst[4 * q + e] = v;
    }
}

template <class EV>
__global__ void __launch_bounds__(EV::NT, 1) ode_rk45_kernel(OdeArgs a) {
    constexpr int RT = EV::RT, NT = EV::NT, XS = EV::XS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typename EV::Smem &S = EV::smem(smem_raw);
    typename EV::Ctx ctx;
    unsigned int gbar_target = 0;
    const int tid = threadIdx.x;
    const float *P = a.P;
    const int N = a.N;
    const double n_total = (double)N * 9.0;
    const long long t_kernel0 = clock64();
    EV::setup(S, ctx, P);
    const int tile0 = EV::tile_first(), tile_step = EV::tile_step();
    float *const tqtab = EV::tq(S);
    float *const xin = EV::xin(S);
    const float *const fo = EV::outp(S);

    const double direction = (a.eps > a.T) ? 1.0 : ((a.eps < a.T) ? -1.0 : 1.0);
    const double t_bound = a.eps;
    // the CTAs of a cluster integrate the same tile redundantly, each on its own copy of the state
    const size_t roff = EV::replica_index(ctx) * a.replica;
    double *ycur = a.y[0] + roff, *ynew = a.y[1] + roff;
    // stage derivatives: K0 holds f(t, y); K0 and K6 trade places when a step is accepted (FSAL)
    double *K0 = a.K[0] + roff, *K6 = a.K[6] + roff;
    double *const K1 = a.K[1] + roff, *const K2 = a.K[2] + roff, *const K3 = a.K[3] + roff, *const K4 = a.K[4] + roff,
                 *const K5 = a.K[5] + roff;
    __shared__ double s_coef[8];  // per stage of the current step: 0.5 g(t_s)^2 ...
    __shared__ float s_std[8];    // ... and sigma(t_s) as the network sees it
    long long cyc_tq = 0, cyc_x = 0, cyc_k = 0, cyc_err = 0;
    double nfev = 0, n_acc = 0, n_rej = 0;
    int next_eval = 0;   // dense output: next requested time
    int status = 0;
    int pbuf = 0;

    // RHS of the rows whose float32 inputs sit in S.x -> K[kdst] (float64), scipy's `fun`
    // RHS of the rows whose float32 inputs sit in S.x -> Kd (float64), scipy's `fun`
    auto stage_eval_c = [&](int tile, int tq_slot, float std, double coef, double *Kd) {
        EV::forward(P, a.proj, S, ctx, tqtab + tq_slot * EV::TQW);
        const long long tk0 = clock64();
        ode_store_k<EV>(fo, Kd, tile, N, std, coef);
        cyc_k += clock64() - tk0;
    };
    auto stage_eval = [&](int tile, int tq_slot, double t_stage, double *Kd) {
        const double g = diffusion_f64(t_stage);
        stage_eval_c(tile, tq_slot, sigma_f32((float)t_stage), 0.5 * (g * g), Kd);
    };
    auto set_obj = [&](int tile) { EV::begin_tile(S, ctx, a.proj, tile * RT, N, a.rpo); };

    // ---- f0 = fun(T, y0), d0, d1 (select_initial_step, common.py:68-134) ----
    double t = a.T;
    if (tid == 0) S.times[0] = (float)t;
    __syncthreads();
    EV::stage_tq(P, S, ctx, 1);
    for (int tile = tile0; tile < a.ntiles; tile += tile_step) {
        const int r0 = tile * RT;
        set_obj(tile);
        for (int i = tid; i < RT * XS; i += NT) {
            const int r = i / XS, c = i - XS * r;
            float v = 0.f;
            if (r0 + r < N && c < 9) {
                const double yv = a.x0[(size_t)(r0 + r) * 9 + c];
                ycur[(size_t)(r0 + r) * 9 + c] = yv;
                if (a.traj) a.traj[(size_t)(r0 + r) * 9 + c] = yv;
                v = (float)yv;
            }
            xin[i] = v;
        }
        __syncthreads();
        stage_eval(tile, 0, t, K0);
        double s0 = 0.0, s1 = 0.0;
        for (int i = tid; i < RT * 9; i += NT) {
            const int r = i / 9;
            if (r0 + r < N) {
                const size_t g = (size_t)r0 * 9 + i;
                const double yv = ycur[g], fv = K0[g];
                const double sc = a.atol + fabs(yv) * a.rtol;
                s0 += (yv / sc) * (yv / sc);
                s1 += (fv / sc) * (fv / sc);
            }
        }
        s0 = block_sum(s0, S.red);
        s1 = block_sum(s1, S.red);
        if (tid == 0) {
            a.part[(pbuf * 3 + 0) * a.ntiles + tile] = s0;
            a.part[(pbuf * 3 + 1) * a.ntiles + tile] = s1;
        }
    }
    nfev += 1;
    grid_barrier(a.gbar, gbar_target);
    const double d0 = sqrt(grid_total(a.part + (pbuf * 3 + 0) * a.ntiles, a.ntiles, S.red) / n_total);
    const double d1 = sqrt(grid_total(a.part + (pbuf * 3 + 1) * a.ntiles, a.ntiles, S.red) / n_total);
    pbuf ^= 1;
    const double interval = fabs(t_bound - a.T);
    double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
    h0 = fmin(h0, interval);

    // ---- f1 = fun(t0 + h0*dir, y0 + h0*dir*f0), d2 ----
    {
        const double t1 = t + h0 * direction;
        if (tid == 0) S.times[0] = (float)t1;
        __syncthreads();
        EV::stage_tq(P, S, ctx, 1);
        for (int tile = tile0; tile < a.ntiles; tile += tile_step) {
            const int r0 = tile * RT;
            set_obj(tile);
            for (int i = tid; i < RT * XS; i += NT) {
                const int r = i / XS, c = i - XS * r;
                float v = 0.f;
                if (r0 + r < N && c < 9) {
                    const size_t g = (size_t)(r0 + r) * 9 + c;
                    v = (float)(ycur[g] + h0 * direction * K0[g]);
                }
                xin[i] = v;
            }
            __syncthreads();
            stage_eval(tile, 0, t1, K1);
            double s2 = 0.0;
            for (int i = tid; i < RT * 9; i += NT) {
                const int r = i / 9;
                if (r0 + r < N) {
                    const size_t g = (size_t)r0 * 9 + i;
                    const double sc = a.atol + fabs(ycur[g]) * a.rtol;
                    const double d = (K1[g] - K0[g]) / sc;
                    s2 += d * d;
                }
            }
            s2 = block_sum(s2, S.red);
            if (tid == 0) a.part[(pbuf * 3 + 0) * a.ntiles + tile] = s2;
        }
        nfev += 1;
        grid_barrier(a.gbar, gbar_target);
    }
    const double d2 = sqrt(grid_total(a.part + (pbuf * 3 + 0) * a.ntiles, a.ntiles, S.red) / n_total) / h0;
    pbuf ^= 1;
    double h1;
    if (d1 <= 1e-15 && d2 <= 1e-15) h1 = fmax(1e-6, h0 * 1e-3);
    else h1 = pow(0.01 / fmax(d1, d2), 1.0 / 5.0);
    double h_abs = fmin(fmin(100.0 * h0, h1), interval);
    const double h_initial = h_abs;
    double h_last = 0.0;

    // ---- main loop (ivp.py while status is None; rk.py _step_impl) ----
    long attempts = 0;
    while (direction * (t - t_bound) < 0.0 && status == 0) {
        const double min_step = 10.0 * fabs(nextafter(t, direction * INFINITY) - t);
        if (h_abs < min_step) h_abs = min_step;  // max_step = inf
        bool step_rejected = false;
        while (true) {
            if (h_abs < min_step) { status = -1; break; }
            if (++attempts > 100000) { status = -2; break; }
            double h = h_abs * direction;
            double t_new = t + h;
            if (direction * (t_new - t_bound) > 0.0) t_new = t_bound;
            h = t_new - t;
            h_abs = fabs(h);

            const long long tq0 = clock64();
            if (tid < 6) {
                const double ts = tid < 5 ? t + c_C[tid + 1] * h : t + h;
                S.times[tid] = (float)ts;
            } else if (tid >= 32 && tid < 38) {   // the stage constants, one thread each (pow() is a long chain)
                const int sI = tid - 32;
                const double ts = sI < 5 ? t + c_C[sI + 1] * h : t + h;
                s_std[sI] = sigma_f32((float)ts);
            } else if (tid >= 64 && tid < 70) {
                const int sI = tid - 64;
                const double ts = sI < 5 ? t + c_C[sI + 1] * h : t + h;
                const double g = diffusion_f64(ts);
                s_coef[sI] = 0.5 * (g * g);
            }
            __syncthreads();
            EV::stage_tq(P, S, ctx, 6);
            cyc_tq += clock64() - tq0;

            for (int tile = tile0; tile < a.ntiles; tile += tile_step) {
                set_obj(tile);
                // rk_step (rk.py:14-78).  The derivative of stage s is written by the input pass of stage s + 1 (and the
                // last one by the error pass), straight from the evaluator's output tile.
                auto fwd = [&](int slot) { EV::forward(P, a.proj, S, ctx, tqtab + slot * EV::TQW); };
                long long tx0 = clock64();
                ode_stage_input<EV, 1>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, N, h, fo, nullptr, 0.f, 0.0);
                cyc_x += clock64() - tx0;
                fwd(0);
                tx0 = clock64();
                ode_stage_input<EV, 2>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, N, h, fo, K1, s_std[0], s_coef[0]);
                cyc_x += clock64() - tx0;
                fwd(1);
                tx0 = clock64();
                ode_stage_input<EV, 3>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, N, h, fo, K2, s_std[1], s_coef[1]);
                cyc_x += clock64() - tx0;
                fwd(2);
                tx0 = clock64();
                ode_stage_input<EV, 4>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, N, h, fo, K3, s_std[2], s_coef[2]);
                cyc_x += clock64() - tx0;
                fwd(3);
                tx0 = clock64();
                ode_stage_input<EV, 5>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, N, h, fo, K4, s_std[3], s_coef[3]);
                cyc_x += clock64() - tx0;
                fwd(4);
                tx0 = clock64();
                ode_stage_input<EV, 6>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, N, h, fo, K5, s_std[4], s_coef[4]);
                cyc_x += clock64() - tx0;
                fwd(5);
                // error estimate (rk.py:139-147)
                const long long te0 = clock64();
                double *traj_slot = (a.traj && (int)n_acc + 1 < a.max_traj) ? a.traj + ((size_t)((int)n_acc + 1) * N) * 9 : nullptr;
                double se = ode_error_part<EV>(ycur, ynew, K0, K1, K2, K3, K4, K5, K6, tile, N, h, a.atol, a.rtol, traj_slot,
                                               fo, s_std[5], s_coef[5]);
                se = block_sum(se, S.red);
                if (tid == 0) a.part[(pbuf * 3 + 0) * a.ntiles + tile] = se;
                cyc_err += clock64() - te0;
            }
            nfev += 6;
            const long long tg0 = clock64();
            grid_barrier(a.gbar, gbar_target);
            const double error_norm = sqrt(grid_total(a.part + (pbuf * 3 + 0) * a.ntiles, a.ntiles, S.red) / n_total);
            pbuf ^= 1;
            cyc_err += clock64() - tg0;
            if (error_norm < 1.0) {
                double factor = (error_norm == 0.0) ? 10.0 : fmin(10.0, 0.9 * pow(error_norm, -0.2));
                if (step_rejected) factor = fmin(1.0, factor);
                h_abs *= factor;
                if (a.t_eval != nullptr) {
                    // t_eval handling of ivp.py: every requested time this step has reached or passed is interpolated
                    // by it.  One CTA per tile writes the shared output; the last point (te == t_bound, x == 1) also
                    // replaces y_new in every CTA's private state: the reference denoises res.y[:, -1].
                    while (next_eval < a.n_eval && direction * (a.t_eval[next_eval] - t_new) <= 0.0) {
                        const double xe = (a.t_eval[next_eval] - t) / h;
                        for (int tile = tile0; tile < a.ntiles; tile += tile_step) {
                            if (EV::writer(ctx))
                                ode_dense_point<EV>(ycur, K0, K1, K2, K3, K4, K5, K6, tile, N, h, xe,
                                                    a.dense + ((size_t)next_eval * N + (size_t)tile * RT) * 9);
                            if (next_eval == a.n_eval - 1 && t_new == t_bound)
                                ode_dense_point<EV>(ycur, K0, K1, K2, K3, K4, K5, K6, tile, N, h, xe,
                                                    ynew + (size_t)tile * RT * 9);
                        }
                        ++next_eval;
                    }
                    __syncthreads();
                }
                // accept: y <- y_new, f <- f_new (FSAL: K[6] becomes K[0]); pointer rotation only
                double *ty = ycur; ycur = ynew; ynew = ty;
                double *tk = K0; K0 = K6; K6 = tk;
                t = t_new;
                h_last = h;
                n_acc += 1;
                break;
            } else {
                // max(MIN_FACTOR, SAFETY * norm ** exponent): python max() keeps 0.2 when the rhs is NaN
                const double f = 0.9 * pow(error_norm, -0.2);
                h_abs *= (f > 0.2) ? f : 0.2;
                step_rejected = true;
                n_rej += 1;
            }
        }
    }

    // ---- denoise (samplers.py:238-249), Gram-Schmidt and centre (:251-257) ----
    {
        const float eps_f = (float)a.eps;
        if (a.denoise) {
            if (tid == 0) S.times[0] = eps_f;
            __syncthreads();
            EV::stage_tq(P, S, ctx, 1);
        }
        for (int tile = tile0; tile < a.ntiles; tile += tile_step) {
            const int r0 = tile * RT;
            if (a.denoise) {
                set_obj(tile);
                for (int i = tid; i < RT * XS; i += NT) {
                    const int r = i / XS, c = i - XS * r;
                    float v = 0.f;
                    if (r0 + r < N && c < 9) v = (float)ycur[(size_t)(r0 + r) * 9 + c];
                    xin[i] = v;
                }
                __syncthreads();
                EV::forward(P, a.proj, S, ctx, tqtab);
            }
            for (int r = tid; r < RT; r += NT) {
                if (r0 + r >= N) continue;
                double v[9];
#pragma unroll
                for (int c = 0; c < 9; ++c) v[c] = ycur[(size_t)(r0 + r) * 9 + c];
                if (a.denoise) {
                    const float std = sigma_f32(eps_f);
                    const float dif = diffusion_f32(eps_f);
                    const float step = (float)((1.0 - a.eps) / a.denoise_steps);
#pragma unroll
                    for (int c = 0; c < 9; ++c) {
                        const float grad = fo[r * XS + c] / (std + 1e-7f);
                        const float drift = 0.f - (dif * dif) * grad;
                        v[c] = v[c] + (double)(drift * step);
                    }
                }
                gram_schmidt6<double>(v);
#pragma unroll
                for (int c = 0; c < 3; ++c) v[6 + c] += (double)a.center[(size_t)(r0 + r) * 3 + c];
                if (status != 0) {   // step-size underflow / attempt cap: the state is not a solution -- poison it in band
#pragma unroll
                    for (int c = 0; c < 9; ++c) v[c] = __longlong_as_double(0x7ff8000000000000LL);
                }
#pragma unroll
                for (int c = 0; c < 9; ++c) a.x_out[(size_t)(r0 + r) * 9 + c] = v[c];
            }
            __syncthreads();
        }
    }
    if (blockIdx.x == 0 && tid == 0) {
        a.stats[GP_STAT_NFEV] = nfev;
        a.stats[GP_STAT_ACCEPTED] = n_acc;
        a.stats[GP_STAT_REJECTED] = n_rej;
        a.stats[GP_STAT_STATUS] = (double)status;
        a.stats[GP_STAT_T_FINAL] = t;
        a.stats[GP_STAT_H_INITIAL] = h_initial;
        a.stats[GP_STAT_H_LAST] = h_last;
        a.stats[14] = (double)(clock64() - t_kernel0);
        a.stats[16] = (double)cyc_tq; a.stats[17] = (double)cyc_x; a.stats[18] = (double)cyc_k; a.stats[19] = (double)cyc_err;
    }
    EV::report(ctx, a.stats);
    EV::teardown(S, ctx);
}

// ------------------------------------------------------------------------------------------
// Per-object step control: every object is integrated as if the sampler had been called with that object alone.
// Object b (rows b*R .. b*R+R-1 of the caller's arrays) is integrated by one CTA (or one cluster) from start to end,
// with its own t, h, error norm, accept / reject sequence and statistics; no grid barrier.  Its rows are split into
// `nsub` consecutive tiles of EV::RT rows (one tile for the tensor-core evaluators, R <= 128; the FFMA evaluator
// uses the tile height a one-object batch call would pick).  In the workspace the object owns nsub whole tiles
// (padded tile b*nsub + j), so the batch kernel's per-tile device functions apply unchanged: they see a batch whose
// rows end R rows into the object's first tile.  Norms are summed exactly as the batch kernel sums them for a batch
// of nsub tiles (per-tile block_sum, then block_sum of the tile partials), so the result is bit-identical to a
// batch call with that object alone on the same evaluator shape.
// ------------------------------------------------------------------------------------------
constexpr int OBJ_MAX_SUB = 16;   // 128 rows in tiles of at least 8 rows

struct OdeObjArgs {
    OdeArgs a;          // N = B * R, rpo = R; traj unused; y / K hold nobj * nsub padded tiles
    int nobj, nsub;
    double *obj_stats;  // [nobj][GP_STAT_COUNT]
    const double *T_obj;    // [nobj] start time of each object (device), or nullptr: a.T for every object
    size_t t_eval_stride;   // doubles between the dense-output grids of consecutive objects (0: one shared grid)
};

template <class EV>
__global__ void __launch_bounds__(EV::NT, 1) ode_rk45_obj_kernel(OdeObjArgs oa) {
    constexpr int RT = EV::RT, NT = EV::NT, XS = EV::XS;
    const OdeArgs &a = oa.a;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typename EV::Smem &S = EV::smem(smem_raw);
    typename EV::Ctx ctx;
    const int tid = threadIdx.x;
    const float *P = a.P;
    const int R = a.rpo, nsub = oa.nsub;
    const double n_total = (double)R * 9.0;
    EV::setup(S, ctx, P);
    float *const tqtab = EV::tq(S);
    float *const xin = EV::xin(S);
    const float *const fo = EV::outp(S);
    const double t_bound = a.eps;
    const size_t roff = EV::replica_index(ctx) * a.replica;
    __shared__ double s_T0;   // start time of the current object
    auto direction_of = [&]() { const double T0 = s_T0; return (a.eps > T0) ? 1.0 : ((a.eps < T0) ? -1.0 : 1.0); };
    __shared__ double s_coef[8];
    __shared__ float s_std[8];
    __shared__ double s_part[3][OBJ_MAX_SUB];   // per-tile partial sums of the current object
    // grid_total() of the batch kernel over this object's tile partials (tid < nsub <= NT: one partial per thread)
    auto total = [&](int k) {
        __syncthreads();
        const double v = tid < nsub ? 0.0 + s_part[k][tid] : 0.0;
        return block_sum(v, S.red);
    };

    for (int b = EV::tile_first(); b < oa.nobj; b += EV::tile_step()) {
        double *ycur = a.y[0] + roff, *ynew = a.y[1] + roff;
        double *K0 = a.K[0] + roff, *K6 = a.K[6] + roff;
        double *const K1 = a.K[1] + roff, *const K2 = a.K[2] + roff, *const K3 = a.K[3] + roff,
                     *const K4 = a.K[4] + roff, *const K5 = a.K[5] + roff;
        // tile j of the object is padded tile b*nsub + j; `Nv` is where the object's rows end in the padded numbering
        const int Nv = b * nsub * RT + R;
        auto set_obj = [&](int j) { EV::begin_tile(S, ctx, a.proj, b * R + j * RT, b * R + R, R); };
        auto stage_eval = [&](int tile, double t_stage, double *Kd) {
            const double g = diffusion_f64(t_stage);
            EV::forward(P, a.proj, S, ctx, tqtab);
            ode_store_k<EV>(fo, Kd, tile, Nv, sigma_f32((float)t_stage), 0.5 * (g * g));
        };
        double nfev = 0, n_acc = 0, n_rej = 0;
        int next_eval = 0;
        int status = 0;
        // The object's start time.  It is kept in shared memory and its direction is derived where it is used, rather
        // than held in registers for the whole object: this kernel runs at its register cap.
        double t = oa.T_obj != nullptr ? oa.T_obj[b] : a.T;
        if (tid == 0) { S.times[0] = (float)t; s_T0 = t; }
        __syncthreads();
        EV::stage_tq(P, S, ctx, 1);
        for (int j = 0; j < nsub; ++j) {
            const int tile = b * nsub + j, r0 = tile * RT, c0 = b * R + j * RT;   // padded / caller's first row
            set_obj(j);
            for (int i = tid; i < RT * XS; i += NT) {
                const int r = i / XS, c = i - XS * r;
                float v = 0.f;
                if (r0 + r < Nv && c < 9) {
                    const double yv = a.x0[(size_t)(c0 + r) * 9 + c];
                    ycur[(size_t)(r0 + r) * 9 + c] = yv;
                    v = (float)yv;
                }
                xin[i] = v;
            }
            __syncthreads();
            stage_eval(tile, t, K0);
            double s0 = 0.0, s1 = 0.0;
            for (int i = tid; i < RT * 9; i += NT) {
                const int r = i / 9;
                if (r0 + r < Nv) {
                    const size_t g = (size_t)r0 * 9 + i;
                    const double yv = ycur[g], fv = K0[g];
                    const double sc = a.atol + fabs(yv) * a.rtol;
                    s0 += (yv / sc) * (yv / sc);
                    s1 += (fv / sc) * (fv / sc);
                }
            }
            s0 = block_sum(s0, S.red);
            s1 = block_sum(s1, S.red);
            if (tid == 0) { s_part[0][j] = s0; s_part[1][j] = s1; }
        }
        nfev += 1;
        const double d0 = sqrt(total(0) / n_total);
        const double d1 = sqrt(total(1) / n_total);
        const double interval = fabs(t_bound - s_T0);
        double h0 = (d0 < 1e-5 || d1 < 1e-5) ? 1e-6 : 0.01 * d0 / d1;
        h0 = fmin(h0, interval);

        // ---- f1 = fun(t0 + h0*dir, y0 + h0*dir*f0), d2 ----
        {
            const double direction = direction_of();
            const double t1 = t + h0 * direction;
            if (tid == 0) S.times[0] = (float)t1;
            __syncthreads();
            EV::stage_tq(P, S, ctx, 1);
            for (int j = 0; j < nsub; ++j) {
                const int tile = b * nsub + j, r0 = tile * RT;
                set_obj(j);
                for (int i = tid; i < RT * XS; i += NT) {
                    const int r = i / XS, c = i - XS * r;
                    float v = 0.f;
                    if (r0 + r < Nv && c < 9) {
                        const size_t g = (size_t)(r0 + r) * 9 + c;
                        v = (float)(ycur[g] + h0 * direction * K0[g]);
                    }
                    xin[i] = v;
                }
                __syncthreads();
                stage_eval(tile, t1, K1);
                double s2 = 0.0;
                for (int i = tid; i < RT * 9; i += NT) {
                    const int r = i / 9;
                    if (r0 + r < Nv) {
                        const size_t g = (size_t)r0 * 9 + i;
                        const double sc = a.atol + fabs(ycur[g]) * a.rtol;
                        const double d = (K1[g] - K0[g]) / sc;
                        s2 += d * d;
                    }
                }
                s2 = block_sum(s2, S.red);
                if (tid == 0) s_part[2][j] = s2;
            }
            nfev += 1;
        }
        const double d2 = sqrt(total(2) / n_total) / h0;
        double h1;
        if (d1 <= 1e-15 && d2 <= 1e-15) h1 = fmax(1e-6, h0 * 1e-3);
        else h1 = pow(0.01 / fmax(d1, d2), 1.0 / 5.0);
        double h_abs = fmin(fmin(100.0 * h0, h1), interval);
        const double h_initial = h_abs;
        double h_last = 0.0;

        // ---- main loop (ivp.py while status is None; rk.py _step_impl) ----
        long attempts = 0;
        while (direction_of() * (t - t_bound) < 0.0 && status == 0) {
            const double direction = direction_of();
            const double min_step = 10.0 * fabs(nextafter(t, direction * INFINITY) - t);
            if (h_abs < min_step) h_abs = min_step;
            bool step_rejected = false;
            while (true) {
                if (h_abs < min_step) { status = -1; break; }
                if (++attempts > 100000) { status = -2; break; }
                double h = h_abs * direction;
                double t_new = t + h;
                if (direction * (t_new - t_bound) > 0.0) t_new = t_bound;
                h = t_new - t;
                h_abs = fabs(h);

                if (tid < 6) {
                    const double ts = tid < 5 ? t + c_C[tid + 1] * h : t + h;
                    S.times[tid] = (float)ts;
                } else if (tid >= 32 && tid < 38) {
                    const int sI = tid - 32;
                    const double ts = sI < 5 ? t + c_C[sI + 1] * h : t + h;
                    s_std[sI] = sigma_f32((float)ts);
                } else if (tid >= 64 && tid < 70) {
                    const int sI = tid - 64;
                    const double ts = sI < 5 ? t + c_C[sI + 1] * h : t + h;
                    const double g = diffusion_f64(ts);
                    s_coef[sI] = 0.5 * (g * g);
                }
                __syncthreads();
                EV::stage_tq(P, S, ctx, 6);

                for (int j = 0; j < nsub; ++j) {
                    const int tile = b * nsub + j;
                    set_obj(j);
                    auto fwd = [&](int slot) { EV::forward(P, a.proj, S, ctx, tqtab + slot * EV::TQW); };
                    ode_stage_input<EV, 1>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, Nv, h, fo, nullptr, 0.f, 0.0);
                    fwd(0);
                    ode_stage_input<EV, 2>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, Nv, h, fo, K1, s_std[0], s_coef[0]);
                    fwd(1);
                    ode_stage_input<EV, 3>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, Nv, h, fo, K2, s_std[1], s_coef[1]);
                    fwd(2);
                    ode_stage_input<EV, 4>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, Nv, h, fo, K3, s_std[2], s_coef[2]);
                    fwd(3);
                    ode_stage_input<EV, 5>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, Nv, h, fo, K4, s_std[3], s_coef[3]);
                    fwd(4);
                    ode_stage_input<EV, 6>(ycur, ynew, K0, K1, K2, K3, K4, K5, xin, tile, Nv, h, fo, K5, s_std[4], s_coef[4]);
                    fwd(5);
                    double se = ode_error_part<EV>(ycur, ynew, K0, K1, K2, K3, K4, K5, K6, tile, Nv, h, a.atol, a.rtol,
                                                   nullptr, fo, s_std[5], s_coef[5]);
                    se = block_sum(se, S.red);
                    if (tid == 0) s_part[0][j] = se;
                }
                nfev += 6;
                const double error_norm = sqrt(total(0) / n_total);
                if (error_norm < 1.0) {
                    double factor = (error_norm == 0.0) ? 10.0 : fmin(10.0, 0.9 * pow(error_norm, -0.2));
                    if (step_rejected) factor = fmin(1.0, factor);
                    h_abs *= factor;
                    if (a.t_eval != nullptr) {
                        const double *const t_eval = a.t_eval + (size_t)b * oa.t_eval_stride;   // the object's grid
                        while (next_eval < a.n_eval && direction * (t_eval[next_eval] - t_new) <= 0.0) {
                            const double xe = (t_eval[next_eval] - t) / h;
                            for (int j = 0; j < nsub; ++j) {
                                const int tile = b * nsub + j;
                                if (EV::writer(ctx))
                                    ode_dense_point<EV>(ycur, K0, K1, K2, K3, K4, K5, K6, tile, Nv, h, xe,
                                                        a.dense + ((size_t)next_eval * a.N + (size_t)b * R + (size_t)j * RT) * 9);
                                if (next_eval == a.n_eval - 1 && t_new == t_bound)
                                    ode_dense_point<EV>(ycur, K0, K1, K2, K3, K4, K5, K6, tile, Nv, h, xe,
                                                        ynew + (size_t)tile * RT * 9);
                            }
                            ++next_eval;
                        }
                        __syncthreads();
                    }
                    double *ty = ycur; ycur = ynew; ynew = ty;
                    double *tk = K0; K0 = K6; K6 = tk;
                    t = t_new;
                    h_last = h;
                    n_acc += 1;
                    break;
                } else {
                    const double f = 0.9 * pow(error_norm, -0.2);
                    h_abs *= (f > 0.2) ? f : 0.2;
                    step_rejected = true;
                    n_rej += 1;
                }
            }
        }

        // ---- denoise (samplers.py:238-249), Gram-Schmidt and centre (:251-257) ----
        const float eps_f = (float)a.eps;
        if (a.denoise) {
            if (tid == 0) S.times[0] = eps_f;
            __syncthreads();
            EV::stage_tq(P, S, ctx, 1);
        }
        for (int j = 0; j < nsub; ++j) {
            const int r0 = (b * nsub + j) * RT, c0 = b * R + j * RT;
            if (a.denoise) {
                set_obj(j);
                for (int i = tid; i < RT * XS; i += NT) {
                    const int r = i / XS, c = i - XS * r;
                    float v = 0.f;
                    if (r0 + r < Nv && c < 9) v = (float)ycur[(size_t)(r0 + r) * 9 + c];
                    xin[i] = v;
                }
                __syncthreads();
                EV::forward(P, a.proj, S, ctx, tqtab);
            }
            for (int r = tid; r < RT; r += NT) {
                if (r0 + r >= Nv) continue;
                double v[9];
#pragma unroll
                for (int c = 0; c < 9; ++c) v[c] = ycur[(size_t)(r0 + r) * 9 + c];
                if (a.denoise) {
                    const float std = sigma_f32(eps_f);
                    const float dif = diffusion_f32(eps_f);
                    const float step = (float)((1.0 - a.eps) / a.denoise_steps);
#pragma unroll
                    for (int c = 0; c < 9; ++c) {
                        const float grad = fo[r * XS + c] / (std + 1e-7f);
                        const float drift = 0.f - (dif * dif) * grad;
                        v[c] = v[c] + (double)(drift * step);
                    }
                }
                gram_schmidt6<double>(v);
#pragma unroll
                for (int c = 0; c < 3; ++c) v[6 + c] += (double)a.center[(size_t)(c0 + r) * 3 + c];
                if (status != 0) {   // this object failed: poison its rows only
#pragma unroll
                    for (int c = 0; c < 9; ++c) v[c] = __longlong_as_double(0x7ff8000000000000LL);
                }
#pragma unroll
                for (int c = 0; c < 9; ++c) a.x_out[(size_t)(c0 + r) * 9 + c] = v[c];
            }
            __syncthreads();
        }
        if (EV::writer(ctx) && tid == 0) {
            double *st = oa.obj_stats + (size_t)b * GP_STAT_COUNT;
            st[GP_STAT_NFEV] = nfev;
            st[GP_STAT_ACCEPTED] = n_acc;
            st[GP_STAT_REJECTED] = n_rej;
            st[GP_STAT_STATUS] = (double)status;
            st[GP_STAT_T_FINAL] = t;
            st[GP_STAT_H_INITIAL] = h_initial;
            st[GP_STAT_H_LAST] = h_last;
        }
    }
    EV::teardown(S, ctx);
}

// Summary of the per-object statistics: nfev = max, accepted / rejected = sums, status = the first non-zero one;
// t_final / h_initial / h_last are those of the first failed object, else of object 0.
__global__ void ode_obj_summary_kernel(const double *__restrict__ obj_stats, int nobj, double *__restrict__ stats) {
    if (threadIdx.x != 0) return;
    double nfev = 0, acc = 0, rej = 0;
    int first = 0;
    bool failed = false;
    for (int b = 0; b < nobj; ++b) {
        const double *st = obj_stats + (size_t)b * GP_STAT_COUNT;
        nfev = fmax(nfev, st[GP_STAT_NFEV]);
        acc += st[GP_STAT_ACCEPTED];
        rej += st[GP_STAT_REJECTED];
        if (!failed && st[GP_STAT_STATUS] != 0.0) { failed = true; first = b; }
    }
    const double *f = obj_stats + (size_t)first * GP_STAT_COUNT;
    stats[GP_STAT_NFEV] = nfev;
    stats[GP_STAT_ACCEPTED] = acc;
    stats[GP_STAT_REJECTED] = rej;
    stats[GP_STAT_STATUS] = f[GP_STAT_STATUS];
    stats[GP_STAT_T_FINAL] = f[GP_STAT_T_FINAL];
    stats[GP_STAT_H_INITIAL] = f[GP_STAT_H_INITIAL];
    stats[GP_STAT_H_LAST] = f[GP_STAT_H_LAST];
}

// xs = normalise(traj) + centre, transposed to [N,S,9]            (samplers.py:251-255)
__global__ void traj_finalize_kernel(const double *__restrict__ traj, const float *__restrict__ center,
                                     int S, int N, double *__restrict__ xs) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)S * N) return;
    const int s = (int)(i / N), r = (int)(i % N);
    double v[9];
#pragma unroll
    for (int c = 0; c < 9; ++c) v[c] = traj[i * 9 + c];
    gram_schmidt6<double>(v);
#pragma unroll
    for (int c = 0; c < 3; ++c) v[6 + c] += (double)center[(size_t)r * 3 + c];
#pragma unroll
    for (int c = 0; c < 9; ++c) xs[((size_t)r * S + s) * 9 + c] = v[c];
}

// ------------------------------------------------------------------------------------------
// predictor-corrector sampler (samplers.py:113-177), float32 like the reference
// ------------------------------------------------------------------------------------------
struct PcArgs {
    const float *P, *proj, *x0, *noise, *center, *time_steps;
    int N, rpo, num_steps;
    double snr;
    float *xs, *mean_x;
    float *x;      // [N][9] state
    double *part;  // [2][ntiles]
    unsigned int *gbar;  // grid barrier counter (zeroed before the launch)
    int ntiles;
};

template <class EV>
__global__ void __launch_bounds__(EV::NT, 1) pc_kernel(PcArgs a) {
    constexpr int RT = EV::RT, NT = EV::NT, XS = EV::XS;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    typename EV::Smem &S = EV::smem(smem_raw);
    typename EV::Ctx ctx;
    unsigned int gbar_target = 0;
    const int tid = threadIdx.x, N = a.N;
    const float *P = a.P;
    EV::setup(S, ctx, P);
    const int tile0 = EV::tile_first(), tile_step = EV::tile_step();
    float *const xin = EV::xin(S);
    const float *const fo = EV::outp(S);
    // grad of this CTA's tiles stays in global scratch between the two halves of a step: reuse
    // mean_x as scratch for grad (it is overwritten with the real mean_x at the end of each step).
    float *grad = a.mean_x;
    const float step_size = a.time_steps[0] - a.time_steps[1];
    const float sqrt_step = sqrtf(step_size);
    int pbuf = 0;
    for (int it = 0; it < a.num_steps; ++it) {
        const float tv = a.time_steps[it];
        if (tid == 0) S.times[0] = tv;
        __syncthreads();
        EV::stage_tq(P, S, ctx, 1);
        const float std = sigma_f32(tv);
        for (int tile = tile0; tile < a.ntiles; tile += tile_step) {
            const int r0 = tile * RT;
            EV::begin_tile(S, ctx, a.proj, r0, N, a.rpo);
            for (int i = tid; i < RT * XS; i += NT) {
                const int r = i / XS, c = i - XS * r;
                float v = 0.f;
                // the state is written by one CTA of the tile's cluster and read by all of them: L2 loads
                if (r0 + r < N && c < 9) v = __ldcg((it == 0 ? a.x0 : a.x) + (size_t)(r0 + r) * 9 + c);
                xin[i] = v;
            }
            __syncthreads();
            EV::forward(P, a.proj, S, ctx, EV::tq(S));
            double sn = 0.0;
            for (int r = tid; r < RT; r += NT) {
                if (r0 + r >= N) continue;
                float ss = 0.f;
#pragma unroll
                for (int c = 0; c < 9; ++c) {
                    const float gv = fo[r * XS + c] / (std + 1e-7f);
                    grad[(size_t)(r0 + r) * 9 + c] = gv;
                    ss += gv * gv;
                }
                sn += (double)sqrtf(ss);
            }
            sn = block_sum(sn, S.red);
            if (tid == 0) a.part[pbuf * a.ntiles + tile] = sn;
            __syncthreads();
        }
        grid_barrier(a.gbar, gbar_target);
        const float grad_norm = (float)(grid_total(a.part + pbuf * a.ntiles, a.ntiles, S.red) / (double)N);
        pbuf ^= 1;
        // langevin_step_size = 2 * (snr * sqrt(9) / grad_norm) ** 2      (samplers.py:143-144).
        // np.float64 / Tensor dispatches to Tensor.__rtruediv__ = reciprocal() * other.
        const float q = (1.0f / grad_norm) * (float)(a.snr * 3.0);
        const float lang = 2.f * (q * q);
        const float sq2l = sqrtf(2.f * lang);
        const float dif = diffusion_f32(tv);
        const float *z1 = a.noise + ((size_t)it * 2 + 0) * N * 9;
        const float *z2 = a.noise + ((size_t)it * 2 + 1) * N * 9;
        for (int tile = tile0; tile < a.ntiles; tile += tile_step) {
            const int r0 = tile * RT;
            // the update overwrites what it reads (state, and grad kept in mean_x): one CTA per tile does it
            for (int r = tid; r < RT && EV::writer(ctx); r += NT) {
                if (r0 + r >= N) continue;
                const size_t g = (size_t)(r0 + r) * 9;
                float x[9], gr[9], m[9];
#pragma unroll
                for (int c = 0; c < 9; ++c) {
                    gr[c] = grad[g + c];
                    const float xv = (it == 0 ? a.x0 : a.x)[g + c];
                    x[c] = (xv + lang * gr[c]) + sq2l * z1[g + c];
                }
                const float na = sqrtf(x[0] * x[0] + x[1] * x[1] + x[2] * x[2]);
                const float nb = sqrtf(x[3] * x[3] + x[4] * x[4] + x[5] * x[5]);
                x[0] /= na; x[1] /= na; x[2] /= na;
                x[3] /= nb; x[4] /= nb; x[5] /= nb;
#pragma unroll
                for (int c = 0; c < 9; ++c) {
                    const float drift = 0.f - (dif * dif) * gr[c];
                    m[c] = x[c] + drift * step_size;
                    x[c] = m[c] + (dif * sqrt_step) * z2[g + c];
                }
                gram_schmidt6<float>(x);
#pragma unroll
                for (int c = 0; c < 9; ++c) a.x[g + c] = x[c];
                if (a.xs) {
#pragma unroll
                    for (int c = 0; c < 9; ++c)
                        a.xs[((size_t)(r0 + r) * a.num_steps + it) * 9 + c] = x[c] + (c >= 6 ? a.center[(size_t)(r0 + r) * 3 + c - 6] : 0.f);
                }
                if (it == a.num_steps - 1) {
#pragma unroll
                    for (int c = 6; c < 9; ++c) m[c] += a.center[(size_t)(r0 + r) * 3 + c - 6];
                    gram_schmidt6<float>(m);
                }
#pragma unroll
                for (int c = 0; c < 9; ++c) a.mean_x[g + c] = m[c];
            }
        }
        __syncthreads();
        EV::tile_sync();
    }
    EV::teardown(S, ctx);
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
// Launch `kern` over tiles: `tiles` CTAs (evaluators without clusters) or `tiles` clusters of EV::CLUSTER CTAs.
// Cooperative launches are clamped to what can be co-resident (tiles are then strided); returns the error code.
template <class EV, class Kern, class Args>
static int launch_tiles(Kern kern, int tiles, bool cooperative, const Args &args, cudaStream_t st, const char *name) {
    const size_t smem = EV::smem_bytes();
    GP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(EV::NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[2];
    int na = 0;
    if (EV::CLUSTER > 1) {
        at[na].id = cudaLaunchAttributeClusterDimension;
        at[na].val.clusterDim.x = EV::CLUSTER; at[na].val.clusterDim.y = 1; at[na].val.clusterDim.z = 1;
        ++na;
    }
    // GP_NONCOOPERATIVE_LAUNCH=1: same grid without the cooperative attribute, for profilers that cannot replay
    // cooperative cluster launches (the grid is still clamped to what is co-resident on an otherwise idle GPU)
    static const bool noncoop = getenv("GP_NONCOOPERATIVE_LAUNCH") && atoi(getenv("GP_NONCOOPERATIVE_LAUNCH")) != 0;
    if (cooperative && !noncoop) {
        at[na].id = cudaLaunchAttributeCooperative;
        at[na].val.cooperative = 1;
        ++na;
    }
    cfg.attrs = at;
    cfg.numAttrs = na;
    int units = tiles;
    if (cooperative) {
        int limit = 0;
        if (EV::CLUSTER > 1) {
            cfg.gridDim = dim3(EV::CLUSTER * tiles);
            if (cudaOccupancyMaxActiveClusters(&limit, kern, &cfg) != cudaSuccess) limit = 0;
        } else {
            int per_sm = 0;
            if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, EV::NT, smem) == cudaSuccess) limit = per_sm * num_sms();
        }
        if (limit <= 0) { set_error("%s: kernel cannot be made resident", name); return GP_ERR_LAUNCH; }
        if (units > limit) units = limit;
    }
    cfg.gridDim = dim3(EV::CLUSTER * units);
    GP_CUDA(cudaLaunchKernelEx(&cfg, kern, args));
    count_launch();
    return GP_OK;
}

static size_t align256(size_t v) { return (v + 255) & ~(size_t)255; }

// Carries an evaluator type to a generic lambda: [&](auto use) { using EV = typename decltype(use)::type; ... }
template <class EV>
struct Use {
    using type = EV;
};

// f(Use<SimtEval<rpt>>{}) for rpt among the FFMA tile heights RPT... the caller instantiates (the last one otherwise)
template <int RPT, int... MORE, class F>
static int with_simt_eval(int rpt, F &f) {
    if constexpr (sizeof...(MORE) == 0) {
        return f(Use<SimtEval<RPT>>{});
    } else {
        return rpt == RPT ? f(Use<SimtEval<RPT>>{}) : with_simt_eval<MORE...>(rpt, f);
    }
}

// The trunk's evaluator for the `mode` of the public entries: calls f(Use<EV>{}) and returns its result.
//   mode & 3       | cluster    | one CTA, A in tensor memory | one CTA, A in shared memory (GP_MODE_SMEM_A)
//   0 fp32 FFMA    | SimtEval<rpt>: the caller's tile rule, one of RPT...; no shapes
//   1 bf16         | TcEval<1>  | TcSoloT<1>                  | TcSolo<1>
//   2 split-bf16   | TcEval<3>  | TcSoloT<3>                  | TcSolo<3>
//   3 tf32         | TcEval<2>  | TcSoloT<2>                  | none: check_mode() refuses it
// GP_MODE_SOLO / GP_MODE_CLUSTER force the shape; by default `shape_rows` that make more 128-row tiles than the GPU
// holds 4-CTA clusters at once (33 on a B200) run one CTA per tile.  `mode` must have passed check_mode().
template <int... RPT, class F>
static int with_evaluator(int mode, int shape_rows, int rpt, F &&f) {
    const bool solo = (mode & GP_MODE_SOLO) || (!(mode & GP_MODE_CLUSTER) && (shape_rows + tc::RT - 1) / tc::RT > 32);
    const bool smem_a = (mode & GP_MODE_SMEM_A) != 0;
    switch (mode & 3) {
        case 1: return !solo ? f(Use<TcEval<1>>{}) : smem_a ? f(Use<TcSolo<1>>{}) : f(Use<TcSoloT<1>>{});
        case 2: return !solo ? f(Use<TcEval<3>>{}) : smem_a ? f(Use<TcSolo<3>>{}) : f(Use<TcSoloT<3>>{});
        case 3: return !solo ? f(Use<TcEval<2>>{}) : f(Use<TcSoloT<2>>{});
        default: return with_simt_eval<RPT...>(rpt, f);
    }
}

// Validation of `mode` shared by the trunk entries: a malformed value is a bad argument; tf32 (3) has evaluators with
// the A operand in tensor memory only, so asking for the shared-memory-A shape is unsupported.  Returns the error code.
static int check_mode(int mode, const char *name) {
    GP_REQUIRE((mode & ~(3 | GP_MODE_SOLO | GP_MODE_CLUSTER | GP_MODE_SMEM_A)) == 0 &&
                   (mode & (GP_MODE_SOLO | GP_MODE_CLUSTER)) != (GP_MODE_SOLO | GP_MODE_CLUSTER),
               "%s: mode must be 0 (fp32 FFMA), 1 (bf16 tcgen05), 2 (split-bf16 x3 tcgen05) or 3 (tf32 tcgen05) "
               "[| GP_MODE_SOLO / GP_MODE_CLUSTER / GP_MODE_SMEM_A]", name);
    if ((mode & 3) == 3 && (mode & GP_MODE_SMEM_A)) {
        set_error("%s: tf32 mode (3) has no shared-memory-A evaluator (GP_MODE_SMEM_A)", name);
        return GP_ERR_UNSUPPORTED;
    }
    return GP_OK;
}

// Rows per compute thread of the FFMA evaluator (tile = 4x that many rows): the choice that minimises the
// per-CTA critical path  waves(tiles / SMs) x rows-per-tile; ties go to the larger tile (fewer weight streams).
static int simt_rows_per_thread(int N, int sms) {
    int best = 8;
    long best_cost = -1;
    for (int rpt = 8; rpt >= 2; rpt -= 2) {
        const long tiles = (N + 4 * rpt - 1) / (4 * rpt);
        const long cost = ((tiles + sms - 1) / sms) * rpt;
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = rpt; }
    }
    return best;
}

}  // namespace gp

using namespace gp;

extern "C" size_t gp_trunk_packed_bytes(void) { return TrunkLayout::END * sizeof(float); }

template <bool TF32>
static int trunk_pack(const gp_trunk_params *raw, void *packed, gp_stream_t s, const char *name) {
    GP_REQUIRE(raw && packed, "%s: null pointer", name);
    GP_REQUIRE(raw->pose_w0 && raw->pose_b0 && raw->pose_w1 && raw->pose_b1 && raw->fourier_w && raw->t_w && raw->t_b,
               "%s: null parameter", name);
    for (int h = 0; h < 3; ++h)
        GP_REQUIRE(raw->head_w0[h] && raw->head_b0[h] && raw->head_w1[h] && raw->head_b1[h], "%s: null head %d", name, h);
    GP_REQUIRE(((uintptr_t)packed & 15) == 0, "%s: packed must be 16-byte aligned", name);
    RawTrunk r;
    r.p = *raw;
    pack_trunk_kernel<TF32><<<num_sms() * 4, 256, 0, as_stream(s)>>>(r, (float *)packed);
    GP_CHECK_LAUNCH(name);
    return GP_OK;
}

extern "C" int gp_trunk_pack(const gp_trunk_params *raw, void *packed, gp_stream_t s) {
    return trunk_pack<false>(raw, packed, s, "gp_trunk_pack");
}

extern "C" int gp_trunk_pack_tf32(const gp_trunk_params *raw, void *packed, gp_stream_t s) {
    return trunk_pack<true>(raw, packed, s, "gp_trunk_pack_tf32");
}

extern "C" int gp_trunk_project(const void *packed, const float *pts_feat, int B, float *proj, gp_stream_t s) {
    GP_REQUIRE(B >= 0, "gp_trunk_project: B < 0");
    if (B == 0) return GP_OK;
    GP_REQUIRE(packed && pts_feat && proj, "gp_trunk_project: null pointer");
    GP_REQUIRE(((uintptr_t)pts_feat & 15) == 0, "gp_trunk_project: pts_feat must be 16-byte aligned");
    dim3 grid(768 / PJ_OUT, (B + PJ_OBJ - 1) / PJ_OBJ);
    project_kernel<<<grid, 256, 0, as_stream(s)>>>((const float *)packed, pts_feat, B, proj);
    GP_CHECK_LAUNCH("gp_trunk_project");
    return GP_OK;
}

// Single evaluation (MODE 0) or energy (MODE 1): FFMA tiles of 16 rows up to 16 rows per SM, 32 above.
template <int MODE>
static int launch_eval(const EvalArgs &a, int mode, cudaStream_t st, const char *name) {
    return with_evaluator<4, 8>(mode, a.N, a.N <= 16 * num_sms() ? 4 : 8, [&](auto use) {
        using EV = typename decltype(use)::type;
        return launch_tiles<EV>(eval_kernel<EV, MODE>, (a.N + EV::RT - 1) / EV::RT, false, a, st, name);
    });
}

extern "C" int gp_scorenet_eval(const void *packed, const float *proj, const float *x, const float *t,
                                int N, int rows_per_object, float *score, int mode, gp_stream_t s) {
    GP_REQUIRE(N >= 0 && rows_per_object >= 1, "gp_scorenet_eval: bad sizes");
    if (N == 0) return GP_OK;
    GP_REQUIRE(packed && proj && x && t && score, "gp_scorenet_eval: null pointer");
    if (const int rc = check_mode(mode, "gp_scorenet_eval")) return rc;
    const EvalArgs a = {(const float *)packed, proj, x, nullptr, nullptr, t, N, rows_per_object, score};
    return launch_eval<0>(a, mode, as_stream(s), "gp_scorenet_eval");
}

extern "C" int gp_energy(const void *packed, const float *proj, const double *poses, const float *pts_center,
                         const float *t_rows, int N, int rows_per_object, float *energy, int mode, gp_stream_t s) {
    GP_REQUIRE(N >= 0 && rows_per_object >= 1, "gp_energy: bad sizes");
    if (N == 0) return GP_OK;
    GP_REQUIRE(packed && proj && poses && pts_center && t_rows && energy, "gp_energy: null pointer");
    if (const int rc = check_mode(mode, "gp_energy")) return rc;
    const EvalArgs a = {(const float *)packed, proj, nullptr, poses, pts_center, t_rows, N, rows_per_object, energy};
    return launch_eval<1>(a, mode, as_stream(s), "gp_energy");
}

// one [N][9] float64 array, padded to whole 128-row tiles (the per-tile vector loads are unconditional)
static size_t ode_state_bytes(int N) { return align256(((size_t)N + 127) / 128 * 128 * 9 * sizeof(double)); }

extern "C" size_t gp_scorenet_ode_workspace_bytes(int N) {
    if (N < 0) return 0;
    const size_t state = ode_state_bytes(N);
    const size_t ntiles_max = (size_t)(N + 7) / 8 + 1;
    return state * 9 * tc::CL + align256(2 * 3 * ntiles_max * sizeof(double)) + 256 /*barrier*/ + 256;
}

// The OdeArgs fields the batch and per-object entries share.  With t_eval (dense output) the denoise step is
// (1 - eps) / n_eval, otherwise (1 - eps) / 1000 (samplers.py:238-249).
static OdeArgs ode_args(const void *packed, const float *proj, const double *x0, const float *pts_center, int N,
                        int rows_per_object, double T, double eps, double rtol, double atol, int denoise,
                        double *x_out, const double *t_eval, int n_eval, double *dense, double *stats) {
    // scipy validate_tol: rtol is clamped to 100 * EPS
    if (rtol < 100 * 2.220446049250313e-16) rtol = 100 * 2.220446049250313e-16;
    OdeArgs a = {};
    a.P = (const float *)packed; a.proj = proj; a.x0 = x0; a.center = pts_center;
    a.N = N; a.rpo = rows_per_object; a.T = T; a.eps = eps; a.rtol = rtol; a.atol = atol;
    a.denoise = denoise; a.x_out = x_out; a.stats = stats;
    a.t_eval = t_eval; a.n_eval = t_eval ? n_eval : 0; a.dense = dense;
    a.denoise_steps = t_eval ? (double)n_eval : 1000.0;
    return a;
}

// y[0..1] and K[0..6], `state` bytes each, from the 256-byte aligned start of the workspace, followed by the copies
// of the other cluster ranks (a.replica doubles apart).  Returns the first byte after them.
static unsigned char *carve_ode_state(OdeArgs &a, void *workspace, size_t state) {
    unsigned char *w = (unsigned char *)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    a.y[0] = (double *)w;
    a.y[1] = (double *)(w + state);
    for (int k = 0; k < 7; ++k) a.K[k] = (double *)(w + (2 + k) * state);
    a.replica = 9 * state / sizeof(double);
    return w + tc::CL * 9 * state;
}

static int scorenet_ode_impl(const void *packed, const float *proj, const double *x0, const float *pts_center,
                             int N, int rows_per_object, double T, double eps, double rtol, double atol,
                             int denoise, double *x_out, double *traj, int max_traj, const double *t_eval, int n_eval,
                             double *dense, double *stats, void *workspace, size_t workspace_bytes, int mode,
                             gp_stream_t s) {
    GP_REQUIRE(packed && proj && x0 && pts_center && x_out && stats && workspace, "gp_scorenet_ode: null pointer");
    GP_REQUIRE(N >= 1 && rows_per_object >= 1, "gp_scorenet_ode: bad sizes N=%d rows_per_object=%d", N, rows_per_object);
    GP_REQUIRE(rtol > 0 && atol > 0, "gp_scorenet_ode: tolerances must be positive");
    GP_REQUIRE(traj == nullptr || max_traj >= 1, "gp_scorenet_ode: max_traj < 1");
    if (const int rc = check_mode(mode, "gp_scorenet_ode")) return rc;
    GP_REQUIRE((t_eval == nullptr) == (dense == nullptr) && (t_eval == nullptr || n_eval >= 1), "gp_scorenet_ode_dense: t_eval / dense / n_eval inconsistent");
    if (workspace_bytes < gp_scorenet_ode_workspace_bytes(N)) {
        set_error("gp_scorenet_ode: workspace too small (%zu < %zu)", workspace_bytes, gp_scorenet_ode_workspace_bytes(N));
        return GP_ERR_WORKSPACE;
    }
    OdeArgs a = ode_args(packed, proj, x0, pts_center, N, rows_per_object, T, eps, rtol, atol, denoise, x_out, t_eval,
                         n_eval, dense, stats);
    a.traj = traj; a.max_traj = max_traj;
    unsigned char *w = carve_ode_state(a, workspace, ode_state_bytes(N));
    a.part = (double *)w; w += align256(2 * 3 * ((size_t)(N + 7) / 8 + 1) * sizeof(double));
    a.gbar = (unsigned int *)w;
    cudaStream_t st = as_stream(s);
    GP_CUDA(cudaMemsetAsync(a.gbar, 0, 256, st));
    return with_evaluator<2, 4, 6, 8>(mode, N, simt_rows_per_thread(N, num_sms()), [&](auto use) {
        using EV = typename decltype(use)::type;
        a.ntiles = (N + EV::RT - 1) / EV::RT;
        return launch_tiles<EV>(ode_rk45_kernel<EV>, a.ntiles, true, a, st, "gp_scorenet_ode");
    });
}

extern "C" int gp_scorenet_ode(const void *packed, const float *proj, const double *x0, const float *pts_center,
                               int N, int rows_per_object, double T, double eps, double rtol, double atol,
                               int denoise, double *x_out, double *traj, int max_traj, double *stats,
                               void *workspace, size_t workspace_bytes, int mode, gp_stream_t s) {
    return scorenet_ode_impl(packed, proj, x0, pts_center, N, rows_per_object, T, eps, rtol, atol, denoise, x_out, traj,
                             max_traj, nullptr, 0, nullptr, stats, workspace, workspace_bytes, mode, s);
}

extern "C" int gp_scorenet_ode_dense(const void *packed, const float *proj, const double *x0, const float *pts_center,
                                     int N, int rows_per_object, double T, double eps, double rtol, double atol,
                                     int denoise, double *x_out, const double *t_eval, int n_eval, double *dense,
                                     double *stats, void *workspace, size_t workspace_bytes, int mode, gp_stream_t s) {
    GP_REQUIRE(t_eval && dense && n_eval >= 1, "gp_scorenet_ode_dense: t_eval / dense missing");
    return scorenet_ode_impl(packed, proj, x0, pts_center, N, rows_per_object, T, eps, rtol, atol, denoise, x_out, nullptr,
                             0, t_eval, n_eval, dense, stats, workspace, workspace_bytes, mode, s);
}

// Per-object step control.  Each object owns 128 padded rows of every state array (one 128-row tile, or whole
// FFMA tiles of at most 128 rows), replicated per cluster rank like the batch workspace.
static size_t ode_obj_state_bytes(int B) { return align256((size_t)B * 128 * 9 * sizeof(double)); }

extern "C" size_t gp_scorenet_ode_objects_workspace_bytes(int B, int R) {
    if (B < 1 || R < 1 || R > 128) return 0;
    return ode_obj_state_bytes(B) * 9 * tc::CL + 256;
}

// T_obj: [B] start times (device), or nullptr for T everywhere; with T_obj the dense-output grid is per object
// ([B][n_eval]), without it one grid serves every object.
static int scorenet_ode_objects_impl(const void *packed, const float *proj, const double *x0, const float *pts_center,
                                     int N, int rows_per_object, double T, const double *T_obj, double eps, double rtol,
                                     double atol, int denoise, double *x_out, const double *t_eval, int n_eval,
                                     double *dense, double *stats, double *obj_stats, void *workspace,
                                     size_t workspace_bytes, int mode, gp_stream_t s) {
    GP_REQUIRE(packed && proj && x0 && pts_center && x_out && stats && obj_stats && workspace,
               "gp_scorenet_ode_objects: null pointer");
    GP_REQUIRE(N >= 1 && rows_per_object >= 1 && N % rows_per_object == 0,
               "gp_scorenet_ode_objects: bad sizes N=%d rows_per_object=%d (N must be B * rows_per_object)", N, rows_per_object);
    if (rows_per_object > 128) {
        set_error("gp_scorenet_ode_objects: rows_per_object=%d > 128 (an object must fit one 128-row tile)", rows_per_object);
        return GP_ERR_UNSUPPORTED;
    }
    GP_REQUIRE(rtol > 0 && atol > 0, "gp_scorenet_ode_objects: tolerances must be positive");
    if (const int rc = check_mode(mode, "gp_scorenet_ode_objects")) return rc;
    GP_REQUIRE((t_eval == nullptr) == (dense == nullptr) && (t_eval == nullptr || n_eval >= 1),
               "gp_scorenet_ode_dense_objects: t_eval / dense / n_eval inconsistent");
    const int B = N / rows_per_object;
    if (workspace_bytes < gp_scorenet_ode_objects_workspace_bytes(B, rows_per_object)) {
        set_error("gp_scorenet_ode_objects: workspace too small (%zu < %zu)", workspace_bytes,
                  gp_scorenet_ode_objects_workspace_bytes(B, rows_per_object));
        return GP_ERR_WORKSPACE;
    }
    OdeObjArgs oa = {};
    oa.a = ode_args(packed, proj, x0, pts_center, N, rows_per_object, T, eps, rtol, atol, denoise, x_out, t_eval, n_eval,
                    dense, stats);
    carve_ode_state(oa.a, workspace, ode_obj_state_bytes(B));
    oa.nobj = B;
    oa.obj_stats = obj_stats;
    oa.T_obj = T_obj;
    oa.t_eval_stride = (T_obj != nullptr && t_eval != nullptr) ? (size_t)n_eval : 0;
    cudaStream_t st = as_stream(s);
    // The evaluator shape follows the tile count B exactly as the batch rule follows its tile count; the FFMA tile
    // height is that of a batch call with this one object, so that the two agree bit for bit.
    const int rpt = simt_rows_per_thread(rows_per_object, num_sms());
    const int rc = with_evaluator<2, 4, 6, 8>(mode, B * tc::RT, rpt, [&](auto use) {
        using EV = typename decltype(use)::type;
        oa.nsub = (rows_per_object + EV::RT - 1) / EV::RT;
        if (oa.nsub * EV::RT > 128 || oa.nsub > OBJ_MAX_SUB) {
            set_error("gp_scorenet_ode_objects: %d rows per object do not fit whole %d-row tiles in 128 rows",
                      rows_per_object, EV::RT);
            return (int)GP_ERR_UNSUPPORTED;
        }
        oa.a.ntiles = B * oa.nsub;
        // One CTA (or cluster) per object, no grid barrier: an ordinary launch whose CTAs the hardware hands out as
        // SMs free up, which balances objects that finish at different step counts.
        return launch_tiles<EV>(ode_rk45_obj_kernel<EV>, B, false, oa, st, "gp_scorenet_ode_objects");
    });
    if (rc != GP_OK) return rc;
    ode_obj_summary_kernel<<<1, 32, 0, st>>>(obj_stats, B, stats);
    GP_CHECK_LAUNCH("gp_scorenet_ode_objects");
    return GP_OK;
}

extern "C" int gp_scorenet_ode_objects(const void *packed, const float *proj, const double *x0, const float *pts_center,
                                       int N, int rows_per_object, double T, double eps, double rtol, double atol,
                                       int denoise, double *x_out, double *stats, double *obj_stats, void *workspace,
                                       size_t workspace_bytes, int mode, gp_stream_t s) {
    return scorenet_ode_objects_impl(packed, proj, x0, pts_center, N, rows_per_object, T, nullptr, eps, rtol, atol,
                                     denoise, x_out, nullptr, 0, nullptr, stats, obj_stats, workspace, workspace_bytes,
                                     mode, s);
}

extern "C" int gp_scorenet_ode_dense_objects(const void *packed, const float *proj, const double *x0,
                                             const float *pts_center, int N, int rows_per_object, double T, double eps,
                                             double rtol, double atol, int denoise, double *x_out, const double *t_eval,
                                             int n_eval, double *dense, double *stats, double *obj_stats,
                                             void *workspace, size_t workspace_bytes, int mode, gp_stream_t s) {
    GP_REQUIRE(t_eval && dense && n_eval >= 1, "gp_scorenet_ode_dense_objects: t_eval / dense missing");
    return scorenet_ode_objects_impl(packed, proj, x0, pts_center, N, rows_per_object, T, nullptr, eps, rtol, atol,
                                     denoise, x_out, t_eval, n_eval, dense, stats, obj_stats, workspace, workspace_bytes,
                                     mode, s);
}

// Per-object start times: T_obj[b] (device; the caller checks T_obj[b] > eps, this entry cannot read it).  t_eval is
// optional and per object, [B][n_eval] in integration order (t_eval[b][0] = T_obj[b]); NULL (with dense NULL) means
// no dense output.
extern "C" int gp_scorenet_ode_objects_t0(const void *packed, const float *proj, const double *x0,
                                          const float *pts_center, int N, int rows_per_object, const double *T_obj,
                                          double eps, double rtol, double atol, int denoise, double *x_out,
                                          const double *t_eval, int n_eval, double *dense, double *stats,
                                          double *obj_stats, void *workspace, size_t workspace_bytes, int mode,
                                          gp_stream_t s) {
    GP_REQUIRE(T_obj, "gp_scorenet_ode_objects_t0: null pointer (T_obj)");
    return scorenet_ode_objects_impl(packed, proj, x0, pts_center, N, rows_per_object, 0.0, T_obj, eps, rtol, atol,
                                     denoise, x_out, t_eval, n_eval, dense, stats, obj_stats, workspace, workspace_bytes,
                                     mode, s);
}

extern "C" int gp_traj_finalize(const double *traj, const float *pts_center, int S, int N, double *xs, gp_stream_t s) {
    GP_REQUIRE(S >= 0 && N >= 0, "gp_traj_finalize: bad sizes");
    if (S == 0 || N == 0) return GP_OK;
    GP_REQUIRE(traj && pts_center && xs, "gp_traj_finalize: null pointer");
    const size_t total = (size_t)S * N;
    traj_finalize_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(s)>>>(traj, pts_center, S, N, xs);
    GP_CHECK_LAUNCH("gp_traj_finalize");
    return GP_OK;
}

extern "C" size_t gp_scorenet_pc_workspace_bytes(int N) {
    if (N < 0) return 0;
    return align256((size_t)N * 9 * sizeof(float)) + align256(2 * ((size_t)(N + 7) / 8 + 1) * sizeof(double)) + 256 /*barrier*/ + 256;
}

extern "C" int gp_scorenet_pc(const void *packed, const float *proj, const float *x0, const float *noise,
                              const float *pts_center, const float *time_steps, int N, int rows_per_object,
                              int num_steps, double snr, float *xs, float *mean_x, void *workspace,
                              size_t workspace_bytes, int mode, gp_stream_t s) {
    GP_REQUIRE(packed && proj && x0 && noise && pts_center && time_steps && mean_x && workspace, "gp_scorenet_pc: null pointer");
    GP_REQUIRE(N >= 1 && rows_per_object >= 1 && num_steps >= 2, "gp_scorenet_pc: bad sizes");
    if (const int rc = check_mode(mode, "gp_scorenet_pc")) return rc;
    if (workspace_bytes < gp_scorenet_pc_workspace_bytes(N)) {
        set_error("gp_scorenet_pc: workspace too small");
        return GP_ERR_WORKSPACE;
    }
    PcArgs a;
    a.P = (const float *)packed; a.proj = proj; a.x0 = x0; a.noise = noise; a.center = pts_center;
    a.time_steps = time_steps; a.N = N; a.rpo = rows_per_object; a.num_steps = num_steps; a.snr = snr;
    a.xs = xs; a.mean_x = mean_x;
    unsigned char *w = (unsigned char *)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
    a.x = (float *)w; w += align256((size_t)N * 9 * sizeof(float));
    a.part = (double *)w; w += align256(2 * ((size_t)(N + 7) / 8 + 1) * sizeof(double));
    a.gbar = (unsigned int *)w;
    cudaStream_t st = as_stream(s);
    GP_CUDA(cudaMemsetAsync(a.gbar, 0, 256, st));
    return with_evaluator<2, 4, 6, 8>(mode, N, simt_rows_per_thread(N, num_sms()), [&](auto use) {
        using EV = typename decltype(use)::type;
        a.ntiles = (N + EV::RT - 1) / EV::RT;
        return launch_tiles<EV>(pc_kernel<EV>, a.ntiles, true, a, st, "gp_scorenet_pc");
    });
}
