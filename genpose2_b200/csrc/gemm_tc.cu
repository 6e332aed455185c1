// Y = relu(X . W^T + b) on the 5th-gen tensor cores (tcgen05 + TMEM), optionally fused with the max-pool
// over `pool_ns` consecutive rows: the SharedMLP layer of a PointNet++ set-abstraction scale
// (P2/pytorch_utils.py:5-33: conv1x1 + BatchNorm(eval, folded) + ReLU; P2/pointnet2_modules.py:59-61)
// on channels-last rows.
//
// Operands are bf16 with fp32 accumulation in TMEM.  NPASS = 1: plain bf16 (bf16 mode).  NPASS = 3: every
// fp32 value is split x = hi + lo (two bf16) and the product is accumulated as hi*hi + lo*hi + hi*lo:
// 16 mantissa bits per operand, relative error ~2^-16 per product -- the fp32-mode encoder path.
// NPASS = 2: tf32 operands rounded to nearest (11 significand bits; tc::tf32_rna_bits), tcgen05.mma.kind::tf32 K = 8.  A 64-k chunk is two
// [rows][32 k] fp32 images (k 0..31, k 32..63) in the slots of the hi and lo images: same bytes, 8 MMAs instead of 12.
//
// CTA = 128 rows x BN (<= 256) columns, K streamed in chunks of 64 through NS shared-memory stages:
//   warps 0-3  A loaders (one row per thread: 16-byte global loads, hi/lo split, swizzled 16-byte smem
//              stores) during the main loop, epilogue afterwards (tcgen05.ld, bias, ReLU, store / pool)
//   warp 4     TMA producer: cp.async.bulk of the pre-packed, pre-swizzled weight chunk images
//   warp 5     MMA issuer: tcgen05.mma.kind::f16 M128 x BN x K16, commits to mbarriers
#include "common.cuh"
#include "tc_ptx.cuh"

namespace gp {
namespace gemm {

constexpr int BM = 128;
constexpr int KC = 64;                   // k per chunk (128 bytes of bf16: one SWIZZLE_128B atom row)
constexpr int A_TILE = BM * 128;         // 16 KB
constexpr int B_TILE_MAX = 256 * 128;    // 32 KB
constexpr int NTHREADS = 192;

struct Args {
    const float *X;        // [R, ldx]
    long long R;
    int ldx;               // floats per row (multiple of 4); columns >= K hold zeros or meet zero weights
    const uint8_t *Wp;     // packed weights
    const float *bias;     // [N]
    int N, K;
    float *Y;              // [R, ldy] or nullptr when pooling
    int ldy;
    int pool_ns;           // 0: no pooling
    float *pooled;         // [R / pool_ns, ld_pooled], zero-initialised by the caller
    int ld_pooled;
    int nchunks;           // ceil(K / 64)
    // gather mode (first SharedMLP layer hoisted to the points, see gp_gemm_gather_bias_relu):
    //   A[r][k] = relu(X[(r / rows_per_batch) * n_src + gidx[r]][k] - Q[r / q_ns][k])
    const int *gidx;       // nullptr: plain mode
    int rows_per_batch, n_src;
    const float *Q;
    int ldq, q_ns;
    int linear;            // 1: epilogue writes X.W^T without bias / ReLU
};

__host__ __device__ inline int bn_of_tile(int N, int j) {  // columns of n-tile j, rounded up to 16
    int rem = N - 256 * j;
    if (rem > 256) rem = 256;
    return (rem + 15) & ~15;
}
__host__ __device__ inline size_t tile_image_bytes(int bn) { return (size_t)bn * 128; }
// packed layout: for n-tile j, for chunk c: hi image [bn x 128 B] then (npass 3) lo image; npass 2: the tf32
// images of k 0..31 and k 32..63
__host__ __device__ inline int images_of(int npass) { return npass == 1 ? 1 : 2; }
__host__ __device__ inline size_t packed_tile_offset(int N, int nchunks, int npass, int j) {
    size_t off = 0;
    const int images = images_of(npass);
    for (int t = 0; t < j; ++t) off += (size_t)nchunks * images * tile_image_bytes(bn_of_tile(N, t));
    return off;
}

__global__ void pack_weights_kernel(const float *__restrict__ W, int N, int K, int npass, int nchunks,
                                    uint8_t *__restrict__ out, size_t total_bytes) {
    // one thread per 4 bytes (two bf16 or one tf32) of the packed buffer
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    const int images = images_of(npass);
    const int ntiles = (N + 255) / 256;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total_bytes / 4; i += stride) {
        size_t o = i * 4;
        int j = 0;
        size_t toff = 0;
        for (; j < ntiles; ++j) {
            const size_t sz = (size_t)nchunks * images * tile_image_bytes(bn_of_tile(N, j));
            if (o < toff + sz) break;
            toff += sz;
        }
        const int bn = bn_of_tile(N, j);
        const size_t img = tile_image_bytes(bn);
        const size_t rel = o - toff;
        const int c = (int)(rel / (images * img));
        const size_t in_c = rel % (images * img);
        const int which = (int)(in_c / img);  // 0 hi, 1 lo (tf32: k 0..31, k 32..63)
        const size_t ob = in_c % img;
        const int nl = (int)(ob / 128), wb = (int)(ob % 128);
        const int logical16 = (wb / 16) ^ (nl & 7);
        const int n = 256 * j + nl;
        if (npass == 2) {   // rounded as the activations are: the MMA would truncate the 13 dropped bits
            const int k = c * KC + which * 32 + logical16 * 4 + (wb % 16) / 4;
            const float w = (n < N && k < K) ? W[(size_t)n * K + k] : 0.f;
            *reinterpret_cast<float *>(out + o) = tc::tf32_rna(w);
            continue;
        }
        const int kk = logical16 * 8 + (wb % 16) / 2;
        float v[2];
        for (int e = 0; e < 2; ++e) {
            const int k = c * KC + kk + e;
            float w = (n < N && k < K) ? W[(size_t)n * K + k] : 0.f;
            const __nv_bfloat16 hi = __float2bfloat16_rn(w);
            v[e] = which == 0 ? __bfloat162float(hi) : (w - __bfloat162float(hi));
        }
        __nv_bfloat162 p = __floats2bfloat162_rn(v[0], v[1]);
        *reinterpret_cast<uint32_t *>(out + o) = *reinterpret_cast<uint32_t *>(&p);
    }
}

// pooled epilogue for one 32-column group: GL lanes form one pooling sub-group
template <int GL>
__device__ __forceinline__ void pool_store(const float (&out)[32], int lane, bool row_ok, long long grow, int ns,
                                           int nbase, const Args &a) {
    constexpr int PER_LANE = 32 / GL;
    const unsigned mask = GL == 32 ? 0xffffffffu : (((1u << GL) - 1u) << ((lane / GL) * GL));
    float keep[PER_LANE];
#pragma unroll
    for (int q = 0; q < PER_LANE; ++q) keep[q] = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
        const unsigned m = redux_max_u32(mask, __float_as_uint(out[j]));
        if ((lane % GL) == (j % GL)) keep[j / GL] = __uint_as_float(m);
    }
    if (row_ok) {
        const long long grp = grow / ns;
#pragma unroll
        for (int q = 0; q < PER_LANE; ++q) {
            const int n = nbase + q * GL + (lane % GL);
            if (n < a.N) {
                float *dst = a.pooled + grp * (long long)a.ld_pooled + n;
                if (ns <= 32) *dst = keep[q];
                else atomicMax(reinterpret_cast<int *>(dst), __float_as_int(keep[q]));
            }
        }
    }
}

// NS_ = shared-memory stages of the K loop.  Grids that cover the GPU at least twice run two CTAs per SM with few
// stages each (the CTAs overlap each other's load / MMA / epilogue phases, which a single CTA executes serially);
// small grids run one CTA per SM with a deeper pipeline.
template <int NPASS, int NS_>
struct Cfg {
    static constexpr int IMAGES = NPASS == 1 ? 1 : 2;
    static constexpr int NS = NS_;
    static constexpr int STAGE_BYTES = IMAGES * (A_TILE + B_TILE_MAX);
    static constexpr size_t SMEM = (size_t)NS * STAGE_BYTES + 1024 /*align*/ + 256 /*barriers*/;
};

template <int NPASS, int NS_>
__global__ void __launch_bounds__(NTHREADS, 2) gemm_bias_relu_kernel(Args a) {
    using C = Cfg<NPASS, NS_>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // pointer arithmetic on the __shared__ array keeps the shared address space (LDS/STS, not generic LD/ST)
    uint8_t *base = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    // stage s: [A_hi | A_lo | B_hi | B_lo]
    auto a_img = [&](int s, int which) { return base + (size_t)s * C::STAGE_BYTES + (size_t)which * A_TILE; };
    auto b_img = [&](int s, int which) { return base + (size_t)s * C::STAGE_BYTES + (size_t)C::IMAGES * A_TILE + (size_t)which * B_TILE_MAX; };
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(base + (size_t)C::NS * C::STAGE_BYTES);
    unsigned long long *a_full = bars, *b_full = bars + C::NS, *empty = bars + 2 * C::NS, *d_full = bars + 3 * C::NS;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 3 * C::NS + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const long long row0 = (long long)blockIdx.x * BM;
    const int jt = blockIdx.y;
    const int bn = bn_of_tile(a.N, jt);
    const int n0 = 256 * jt;

    if (tid == 0) {
        for (int s = 0; s < C::NS; ++s) {
            tc::mbar_init(&a_full[s], 4);   // one elected lane per loader warp
            tc::mbar_init(&b_full[s], 1);
            tc::mbar_init(&empty[s], 1);
        }
        tc::mbar_init(d_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (warp == 5) tc::tmem_alloc(tmem_slot, 256);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem = *tmem_slot;

    if (warp < 4) {
        // ------------------------- A loaders -------------------------
        // Coalesced: in pass i a warp reads two rows' 256-byte chunks (lanes 0-15 row 2i, lanes 16-31 row 2i+1,
        // 16 bytes per lane = 4 full 128-byte lines per instruction), converts its 4 floats to bf16 hi (+ lo)
        // and writes 8 bytes into the swizzled operand row.
        const int jv = lane & 15;                         // 16-byte vector inside the 256-byte chunk
        const int sub = lane >> 4;                        // which of the two rows of this pass
        const int r = tid;                                // epilogue row (TMEM lane) of this thread
        const long long grow = row0 + r;
        const bool row_ok = grow < a.R;
        // register double buffering: the global loads of chunk c+1 are in flight while chunk c is converted
        // (the rows come from HBM; without this the loader is latency bound)
        const bool gather = a.gidx != nullptr;
        // per pass: element offset of the source row in X (-1: no row) and of the group's row in Q, computed once
        // per tile with 32-bit divisions (the host checks that the offsets fit)
        long long src[16];
        int qoff[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) {
            const long long lr = row0 + 32 * warp + 2 * i + sub;
            src[i] = -1;
            qoff[i] = -1;
            if (lr < a.R) {
                const int lr32 = (int)lr;
                const long long srow = gather ? (long long)(lr32 / a.rows_per_batch) * a.n_src + __ldg(a.gidx + lr) : lr;
                src[i] = srow * a.ldx;
                if (gather) qoff[i] = (lr32 / a.q_ns) * a.ldq;
            }
        }
        auto load_chunk = [&](int c, float4 (&v)[16]) {
            const int k = c * KC + 4 * jv;
            const bool k_ok = k < a.ldx;
#pragma unroll
            for (int i = 0; i < 16; ++i)
                v[i] = (k_ok && src[i] >= 0) ? __ldg(reinterpret_cast<const float4 *>(a.X + src[i] + k))
                                             : make_float4(0.f, 0.f, 0.f, 0.f);
        };
        auto convert_store = [&](int s, int cc, const float4 (&v)[16]) {
            uint8_t *hi_img = a_img(s, 0), *lo_img = a_img(s, 1);
#pragma unroll
            for (int i = 0; i < 16; ++i) {
                const int rl = 32 * warp + 2 * i + sub;   // row inside the tile
                const int off = rl * 128 + (((jv >> 1) ^ (rl & 7)) << 4) + ((jv & 1) << 3);
                float4 p = v[i];
                if (gather) {  // hoisted first layer: relu(P[src] - Q[group]); Q rows hit L1 (shared by q_ns rows)
                    const int k = cc * KC + 4 * jv;
                    if (qoff[i] >= 0 && k < a.ldq) {
                        const float4 q = __ldg(reinterpret_cast<const float4 *>(a.Q + qoff[i] + k));
                        p.x = fmaxf(p.x - q.x, 0.f); p.y = fmaxf(p.y - q.y, 0.f);
                        p.z = fmaxf(p.z - q.z, 0.f); p.w = fmaxf(p.w - q.w, 0.f);
                    } else {
                        p = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                if (NPASS == 2) {
                    // 16 bytes = k 4 jv .. 4 jv + 3: image jv / 8, 16-byte unit jv % 8 of its 128-byte row
                    const int toff = rl * 128 + (((jv & 7) ^ (rl & 7)) << 4);
                    const uint4 t = make_uint4(tc::tf32_rna_bits(p.x), tc::tf32_rna_bits(p.y), tc::tf32_rna_bits(p.z),
                                               tc::tf32_rna_bits(p.w));
                    *reinterpret_cast<uint4 *>((jv < 8 ? hi_img : lo_img) + toff) = t;
                    continue;
                }
                const __nv_bfloat162 h0 = __floats2bfloat162_rn(p.x, p.y), h1 = __floats2bfloat162_rn(p.z, p.w);
                uint2 pk;
                pk.x = *reinterpret_cast<const uint32_t *>(&h0); pk.y = *reinterpret_cast<const uint32_t *>(&h1);
                *reinterpret_cast<uint2 *>(hi_img + off) = pk;
                if (NPASS == 3) {
                    const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
                    const __nv_bfloat162 l0 = __floats2bfloat162_rn(p.x - f0.x, p.y - f0.y);
                    const __nv_bfloat162 l1 = __floats2bfloat162_rn(p.z - f1.x, p.w - f1.y);
                    uint2 pl;
                    pl.x = *reinterpret_cast<const uint32_t *>(&l0); pl.y = *reinterpret_cast<const uint32_t *>(&l1);
                    *reinterpret_cast<uint2 *>(lo_img + off) = pl;
                }
            }
        };
        float4 va[16];
        for (int c = 0; c < a.nchunks; ++c) {
            load_chunk(c, va);
            const int s = c % C::NS;
            if (c >= C::NS) tc::mbar_wait(&empty[s], ((c / C::NS) + 1) & 1);
            convert_store(s, c, va);
            tc::fence_proxy_async();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&a_full[s]);
        }
        // ------------------------- epilogue -------------------------
        tc::mbar_wait(d_full, 0);
        tc::tc_fence_after();
        const uint32_t lane_addr = tmem + ((uint32_t)(32 * warp) << 16);
        const int ns = a.pool_ns;
        for (int g = 0; g < bn / 32 + ((bn & 31) ? 1 : 0); ++g) {
            uint32_t rv[32];
            tc::tmem_ld32(lane_addr + g * 32, rv);
            float out[32];
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                const int n = n0 + g * 32 + j;
                const float bv = (n < a.N && !a.linear) ? __ldg(a.bias + n) : 0.f;
                const float acc = __uint_as_float(rv[j]) + bv;
                out[j] = (n < a.N && row_ok) ? (a.linear ? acc : fmaxf(acc, 0.f)) : 0.f;
            }
            if (ns == 0) {
                // transpose the warp's 32 x 32 block through shared memory (the operand stages are free once
                // d_full has fired) so that every store instruction writes one full 128-byte line of one row
                float *stg = reinterpret_cast<float *>(base) + warp * (32 * 33);
#pragma unroll
                for (int j = 0; j < 32; ++j) stg[lane * 33 + j] = out[j];
                __syncwarp();
                const int ncol = n0 + g * 32 + lane;
                if (ncol < a.ldy) {
                    const long long rbase = row0 + 32 * warp;
#pragma unroll 4
                    for (int rr = 0; rr < 32; ++rr)
                        if (rbase + rr < a.R) a.Y[(rbase + rr) * (long long)a.ldy + ncol] = stg[rr * 33 + lane];
                }
                __syncwarp();
            } else {
                // max over the pool_ns consecutive rows of each group.  Values are >= 0 after the ReLU, so the
                // float order equals the unsigned order of the bit patterns: one redux.sync per column.
                if (ns >= 32) pool_store<32>(out, lane, row_ok, grow, ns, n0 + g * 32, a);
                else if (ns == 16) pool_store<16>(out, lane, row_ok, grow, ns, n0 + g * 32, a);
                else pool_store<8>(out, lane, row_ok, grow, ns, n0 + g * 32, a);
            }
        }
        tc::tc_fence_before();
    } else if (warp == 4) {
        // ------------------------- TMA producer (weights) -------------------------
        if (lane == 0) {
            const size_t img = tile_image_bytes(bn);
            const uint8_t *src = a.Wp + packed_tile_offset(a.N, a.nchunks, NPASS, jt);
            for (int c = 0; c < a.nchunks; ++c) {
                const int s = c % C::NS;
                if (c >= C::NS) tc::mbar_wait(&empty[s], ((c / C::NS) + 1) & 1);
                tc::mbar_arrive_expect_tx(&b_full[s], (uint32_t)(C::IMAGES * img));
                for (int w = 0; w < C::IMAGES; ++w)
                    tc::bulk_g2s(b_img(s, w), src + ((size_t)c * C::IMAGES + w) * img, (uint32_t)img, &b_full[s]);
            }
        }
        __syncwarp();
    } else {
        // ------------------------- MMA issuer -------------------------
        if (lane == 0) {
            const uint32_t idesc = NPASS == 2 ? tc::make_idesc_tf32(128, (uint32_t)bn) : tc::make_idesc_bf16(128, (uint32_t)bn);
            for (int c = 0; c < a.nchunks; ++c) {
                const int s = c % C::NS;
                const uint32_t ph = (c / C::NS) & 1;
                tc::mbar_wait(&a_full[s], ph);
                tc::mbar_wait(&b_full[s], ph);
                tc::tc_fence_after();
                const uint32_t ahi = tc::smem_u32(a_img(s, 0)), alo = tc::smem_u32(a_img(s, 1));
                const uint32_t bhi = tc::smem_u32(b_img(s, 0)), blo = tc::smem_u32(b_img(s, 1));
                if (NPASS == 2) {
#pragma unroll
                    for (int kk = 0; kk < 8; ++kk) {   // K = 8 steps: 4 in the image of k 0..31, 4 in that of k 32..63
                        const uint32_t ao = (kk < 4 ? ahi : alo) + (kk & 3) * 32, bo = (kk < 4 ? bhi : blo) + (kk & 3) * 32;
                        tc::umma_tf32_ss(tmem, tc::make_desc(ao), tc::make_desc(bo), idesc, (c | kk) ? 1u : 0u);
                    }
                }
#pragma unroll
                for (int kk = 0; kk < (NPASS == 2 ? 0 : 4); ++kk) {
                    tc::umma_bf16(tmem, tc::make_desc(ahi + kk * 32), tc::make_desc(bhi + kk * 32), idesc, (c | kk) ? 1u : 0u);
                    if (NPASS == 3) {
                        tc::umma_bf16(tmem, tc::make_desc(alo + kk * 32), tc::make_desc(bhi + kk * 32), idesc, 1u);
                        tc::umma_bf16(tmem, tc::make_desc(ahi + kk * 32), tc::make_desc(blo + kk * 32), idesc, 1u);
                    }
                }
                tc::umma_commit(&empty[s]);
            }
            tc::umma_commit(d_full);
        }
        __syncwarp();
    }
    __syncthreads();
    if (warp == 5) tc::tmem_dealloc(tmem, 256);
}

template <int NPASS, int NS_>
static int launch_ns(const Args &a, cudaStream_t st) {
    auto kern = gemm_bias_relu_kernel<NPASS, NS_>;
    GP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)Cfg<NPASS, NS_>::SMEM));
    dim3 grid((unsigned)((a.R + BM - 1) / BM), (unsigned)((a.N + 255) / 256));
    kern<<<grid, NTHREADS, Cfg<NPASS, NS_>::SMEM, st>>>(a);
    GP_CHECK_LAUNCH("gp_gemm_bias_relu");
    return GP_OK;
}

template <int NPASS>
static int launch(const Args &a, cudaStream_t st) {
    const long long ctas = ((a.R + BM - 1) / BM) * ((a.N + 255) / 256);
    const bool wide = ctas >= 2LL * num_sms();
    // split-bf16 and tf32: a stage is 96 KB (one per CTA when two CTAs share an SM, two otherwise); bf16: 48 KB (two / four)
    if (NPASS != 1) return wide ? launch_ns<NPASS, 1>(a, st) : launch_ns<NPASS, 2>(a, st);
    return wide ? launch_ns<NPASS, 2>(a, st) : launch_ns<NPASS, 4>(a, st);
}

static int launch_npass(const Args &a, int npass, cudaStream_t st) {
    return npass == 3 ? launch<3>(a, st) : npass == 2 ? launch<2>(a, st) : launch<1>(a, st);
}

}  // namespace gemm
}  // namespace gp

using namespace gp;

extern "C" size_t gp_gemm_packed_bytes(int N, int K, int npass) {
    if (N < 1 || K < 1 || npass < 1 || npass > 3) return 0;
    const int nchunks = (K + gemm::KC - 1) / gemm::KC;
    return gemm::packed_tile_offset(N, nchunks, npass, (N + 255) / 256);
}

extern "C" int gp_gemm_pack(const float *W, int N, int K, int npass, void *packed, gp_stream_t s) {
    GP_REQUIRE(W && packed, "gp_gemm_pack: null pointer");
    GP_REQUIRE(N >= 1 && K >= 1 && npass >= 1 && npass <= 3, "gp_gemm_pack: bad arguments (npass must be 1, 2 or 3)");
    GP_REQUIRE(((uintptr_t)packed & 15) == 0, "gp_gemm_pack: packed must be 16-byte aligned");
    const int nchunks = (K + gemm::KC - 1) / gemm::KC;
    const size_t total = gp_gemm_packed_bytes(N, K, npass);
    gemm::pack_weights_kernel<<<num_sms() * 4, 256, 0, as_stream(s)>>>(W, N, K, npass, nchunks, (uint8_t *)packed, total);
    GP_CHECK_LAUNCH("gp_gemm_pack");
    return GP_OK;
}

extern "C" int gp_gemm_bias_relu(const float *X, long long R, int ldx, const void *packed, const float *bias, int N,
                                 int K, int npass, float *Y, int ldy, int pool_ns, float *pooled, int ld_pooled,
                                 gp_stream_t s) {
    GP_REQUIRE(R >= 0 && N >= 1 && K >= 1 && npass >= 1 && npass <= 3, "gp_gemm_bias_relu: bad arguments (npass must be 1, 2 or 3)");
    if (R == 0) return GP_OK;
    GP_REQUIRE(X && packed && bias, "gp_gemm_bias_relu: null pointer");
    GP_REQUIRE(ldx >= 4 && (ldx & 3) == 0 && ((uintptr_t)X & 15) == 0, "gp_gemm_bias_relu: X rows must be 16-byte aligned (ldx %% 4 == 0)");
    GP_REQUIRE(((uintptr_t)packed & 15) == 0, "gp_gemm_bias_relu: packed must be 16-byte aligned");
    if (pool_ns == 0) {
        GP_REQUIRE(Y && ldy >= N && ldy <= ((N + 31) & ~31) && (ldy & 3) == 0 && ((uintptr_t)Y & 15) == 0,
                   "gp_gemm_bias_relu: bad Y / ldy (need N <= ldy <= round_up(N, 32), ldy %% 4 == 0)");
    } else {
        GP_REQUIRE(pooled && ld_pooled >= N, "gp_gemm_bias_relu: bad pooled output");
        GP_REQUIRE(pool_ns >= 1 && ((pool_ns <= 32 && 32 % pool_ns == 0) || pool_ns % 32 == 0) && R % pool_ns == 0,
                   "gp_gemm_bias_relu: pool_ns=%d must divide 32 or be a multiple of 32, and divide R", pool_ns);
        GP_REQUIRE(pool_ns == 8 || pool_ns == 16 || pool_ns % 32 == 0, "gp_gemm_bias_relu: pool_ns must be 8, 16 or a multiple of 32");
    }
    gemm::Args a;
    a.X = X; a.R = R; a.ldx = ldx; a.Wp = (const uint8_t *)packed; a.bias = bias; a.N = N; a.K = K;
    a.Y = Y; a.ldy = ldy; a.pool_ns = pool_ns; a.pooled = pooled; a.ld_pooled = ld_pooled;
    a.nchunks = (K + gemm::KC - 1) / gemm::KC;
    a.gidx = nullptr; a.rows_per_batch = 1; a.n_src = 0; a.Q = nullptr; a.ldq = 0; a.q_ns = 1; a.linear = 0;
    return gemm::launch_npass(a, npass, as_stream(s));
}

extern "C" int gp_gemm_linear(const float *X, long long R, int ldx, const void *packed, int N, int K, int npass,
                              float *Y, int ldy, gp_stream_t s) {
    GP_REQUIRE(R >= 0 && N >= 1 && K >= 1 && npass >= 1 && npass <= 3, "gp_gemm_linear: bad arguments (npass must be 1, 2 or 3)");
    if (R == 0) return GP_OK;
    GP_REQUIRE(X && packed && Y, "gp_gemm_linear: null pointer");
    GP_REQUIRE(ldx >= 4 && (ldx & 3) == 0 && ((uintptr_t)X & 15) == 0, "gp_gemm_linear: X rows must be 16-byte aligned");
    GP_REQUIRE(ldy >= N && ldy <= ((N + 31) & ~31) && (ldy & 3) == 0 && ((uintptr_t)Y & 15) == 0, "gp_gemm_linear: bad Y / ldy");
    gemm::Args a;
    a.X = X; a.R = R; a.ldx = ldx; a.Wp = (const uint8_t *)packed; a.bias = nullptr; a.N = N; a.K = K;
    a.Y = Y; a.ldy = ldy; a.pool_ns = 0; a.pooled = nullptr; a.ld_pooled = 0;
    a.nchunks = (K + gemm::KC - 1) / gemm::KC;
    a.gidx = nullptr; a.rows_per_batch = 1; a.n_src = 0; a.Q = nullptr; a.ldq = 0; a.q_ns = 1; a.linear = 1;
    return gemm::launch_npass(a, npass, as_stream(s));
}

namespace gp {
namespace gemm {
// Q[r][k] = sum_j xyz[r][j] * Wt[j][k] - b[k] for k < c1, zero up to ldq: the per-centre term of a hoisted first layer
__global__ void centre_term_kernel(const float *__restrict__ xyz, long long rows, const float *__restrict__ Wt,
                                   const float *__restrict__ b, int c1, float *__restrict__ Q, int ldq,
                                   const float *__restrict__ tail_src, float *__restrict__ tail_dst, int ld_tail) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= rows * ldq) return;
    const long long r = i / ldq;
    const int k = (int)(i - r * ldq);
    // by-product: the centre's [x y z 0] row into the tail of this level's buffer
    if (tail_dst && k < 4) tail_dst[r * ld_tail + k] = __ldg(tail_src + r * 4 + k);
    float v = 0.f;
    if (k < c1) {
        const float x = __ldg(xyz + r * 3), y = __ldg(xyz + r * 3 + 1), z = __ldg(xyz + r * 3 + 2);
        // the order of torch.addmm's K = 3 dot product does not matter at this size; written as one chain
        v = fmaf(z, __ldg(Wt + 2 * c1 + k), fmaf(y, __ldg(Wt + c1 + k), x * __ldg(Wt + k))) - __ldg(b + k);
    }
    Q[i] = v;
}
}  // namespace gemm
}  // namespace gp

extern "C" int gp_centre_term(const float *new_xyz, long long rows, const float *w0_xyz_t, const float *b0, int c1,
                              float *Q, int ldq, gp_stream_t s) {
    GP_REQUIRE(rows >= 0 && c1 >= 1 && ldq >= c1, "gp_centre_term: bad sizes");
    if (rows == 0) return GP_OK;
    GP_REQUIRE(new_xyz && w0_xyz_t && b0 && Q, "gp_centre_term: null pointer");
    const long long total = rows * ldq;
    gemm::centre_term_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(s)>>>(new_xyz, rows, w0_xyz_t, b0, c1, Q, ldq,
                                                                                            nullptr, nullptr, 0);
    GP_CHECK_LAUNCH("gp_centre_term");
    return GP_OK;
}

extern "C" int gp_centre_term_tail(const float *new_xyz, long long rows, const float *w0_xyz_t, const float *b0, int c1,
                                   float *Q, int ldq, const float *tail_src, float *tail_dst, int ld_tail, gp_stream_t s) {
    GP_REQUIRE(rows >= 0 && c1 >= 1 && ldq >= c1 && ldq >= 4, "gp_centre_term_tail: bad sizes");
    if (rows == 0) return GP_OK;
    GP_REQUIRE(new_xyz && w0_xyz_t && b0 && Q && tail_src && tail_dst && ld_tail >= 4, "gp_centre_term_tail: null pointer");
    const long long total = rows * ldq;
    gemm::centre_term_kernel<<<(unsigned)((total + 255) / 256), 256, 0, as_stream(s)>>>(new_xyz, rows, w0_xyz_t, b0, c1, Q, ldq,
                                                                                            tail_src, tail_dst, ld_tail);
    GP_CHECK_LAUNCH("gp_centre_term_tail");
    return GP_OK;
}

extern "C" int gp_gemm_gather_bias_relu(const float *P, int n_src, int ldp, const int32_t *gidx, long long R,
                                        int rows_per_batch, const float *Q, int ldq, int q_ns, const void *packed,
                                        const float *bias, int N, int K, int npass, float *Y, int ldy, int pool_ns,
                                        float *pooled, int ld_pooled, gp_stream_t s) {
    GP_REQUIRE(R >= 0 && N >= 1 && K >= 1 && npass >= 1 && npass <= 3, "gp_gemm_gather_bias_relu: bad arguments (npass must be 1, 2 or 3)");
    if (R == 0) return GP_OK;
    GP_REQUIRE(P && gidx && Q && packed && bias, "gp_gemm_gather_bias_relu: null pointer");
    GP_REQUIRE(ldp >= 4 && (ldp & 3) == 0 && ((uintptr_t)P & 15) == 0 && ldq >= 4 && (ldq & 3) == 0 && ((uintptr_t)Q & 15) == 0,
               "gp_gemm_gather_bias_relu: P / Q rows must be 16-byte aligned");
    GP_REQUIRE(ldq >= K && ldp >= K, "gp_gemm_gather_bias_relu: ldp and ldq must cover K");
    GP_REQUIRE(rows_per_batch >= 1 && n_src >= 1 && q_ns >= 1, "gp_gemm_gather_bias_relu: bad gather geometry");
    GP_REQUIRE(R < 2147483647LL && (R / q_ns + 1) * (long long)ldq < 2147483647LL, "gp_gemm_gather_bias_relu: too many rows");
    if (pool_ns == 0) {
        GP_REQUIRE(Y && ldy >= N && ldy <= ((N + 31) & ~31) && (ldy & 3) == 0 && ((uintptr_t)Y & 15) == 0,
                   "gp_gemm_gather_bias_relu: bad Y / ldy");
    } else {
        GP_REQUIRE(pooled && ld_pooled >= N && R % pool_ns == 0 && (pool_ns == 8 || pool_ns == 16 || pool_ns % 32 == 0),
                   "gp_gemm_gather_bias_relu: bad pooled output / pool_ns");
    }
    gemm::Args a;
    a.X = P; a.R = R; a.ldx = ldp; a.Wp = (const uint8_t *)packed; a.bias = bias; a.N = N; a.K = K;
    a.Y = Y; a.ldy = ldy; a.pool_ns = pool_ns; a.pooled = pooled; a.ld_pooled = ld_pooled;
    a.nchunks = (K + gemm::KC - 1) / gemm::KC;
    a.gidx = gidx; a.rows_per_batch = rows_per_batch; a.n_src = n_src; a.Q = Q; a.ldq = ldq; a.q_ns = q_ns; a.linear = 0;
    return gemm::launch_npass(a, npass, as_stream(s));
}
