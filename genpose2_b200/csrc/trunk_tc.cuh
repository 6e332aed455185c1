// Tensor-core (tcgen05 + TMEM + TMA bulk copies) tile evaluator of the ScoreNet trunk, cluster edition.
//
// A tile is 128 rows (hypotheses) = one UMMA M=128 accumulator.  A thread-block cluster of CL = 4 CTAs works
// on one tile: every CTA evaluates the (small) pose encoder 9 -> 256 -> 256 for all 128 rows, and the three
// 256 -> 256 head layers -- three quarters of the multiply-adds and of the epilogue work -- are split by output
// column: CTA r owns columns 64r..64r+63 of every head, applies bias / ReLU / the 256 -> 3 output layer to
// them and scatters its [128][9] partial result into the shared memory of all four CTAs (st.shared::cluster).
// After one cluster barrier every CTA holds the same f_theta for the whole tile, bit for bit, so the
// integrator code around it runs replicated and needs no further exchange.  With 25 tiles (64 objects x 50
// hypotheses) this occupies 100 SMs instead of 25 and shortens the per-evaluation critical path ~3x.
//
// Per CTA, 10 warps:
//   warp 0      TMA producer : streams the 16 weight chunks of an evaluation ([128 rows][64 k] bf16 images,
//                              pre-swizzled in global, 16 KB each, L2 resident) through a shared-memory
//                              ring with cp.async.bulk + mbarrier complete_tx, running ahead across
//                              layers and evaluations
//   warp 1      MMA issuer   : one lane issues tcgen05.mma chains (M128, N128 for the encoder, N64 for the
//                              head slices, K16), accumulators in TMEM, commits to mbarriers
//   warps 2..9  epilogue     : 256 threads.  Inputs -> bf16 A operand; TMEM -> registers (tcgen05.ld), bias,
//                              ReLU, bf16 (hi / lo) re-pack into the A operand, which lives in TENSOR MEMORY
//                              (tcgen05.st; the MMAs read it from there): no A buffer in shared memory, so the
//                              weight ring is 5-6 stages deep; heads: + proj + tq from shared memory, ReLU,
//                              256 -> 3 output layer, cluster exchange.
// TMEM map: columns 0..127 A hi (256 k as packed bf16 pairs), 128..255 A lo, 256..511 accumulators (D0 / D1: N = 256;
// heads: N = 192).
//
// NPASS = 1 ("bf16" mode): operands rounded to bf16.
// NPASS = 3 ("fp32" mode): every operand is split x = hi + lo (two bf16) and each product is accumulated as
//   hi*hi + lo*hi + hi*lo in fp32 (TMEM): 16 mantissa bits per operand.  On the reference's own fixtures this
//   is indistinguishable from a plain fp32 evaluation (same size as changing the fp32 summation order),
//   while plain bf16 costs 1e-3 rad / 3e-4.
// NPASS = 2 ("tf32" mode): operands rounded to tf32 (cvt.rna, 11 significand bits), kind::tf32 MMAs of K = 8.  A tf32
//   value is as wide as a hi + lo bf16 pair, so the layout is the split mode's: a chunk's two images hold k 0..31 and
//   k 32..63 in the hi and lo slots of the ring, the A operand fills TMEM columns 0..255 (column = k), and a K = 8 step
//   advances the descriptors by the bytes and columns of a K = 16 bf16 step: 2 MMAs per 16 k instead of 3.
//
// Per evaluation: D0 = x . W1^T ; h1 = relu(D0 + b1) ; D1 = h1 . W2^T ; h2 = relu(D1 + b2) ;
// D2_h = h2 . Whp_h[64r..64r+63]^T (3 heads).  Operand layout: canonical K-major SWIZZLE_128B (8-row x
// 128-byte atoms, 16-byte chunk index XOR row % 8).
#pragma once
#include <cuda_bf16.h>

#include "tc_ptx.cuh"
#include "trunk.cuh"

namespace gp {
namespace tc {

constexpr int RT = 128;               // rows per tile (UMMA M)
constexpr int NTHREADS = 320;         // 10 warps
constexpr int CL = 4;                 // CTAs per cluster
constexpr int HC = 256 / CL;          // head columns owned by one CTA (per head)
constexpr int NHC = 3 * HC;           // ... over the three heads
constexpr int XS = 9;                 // row stride of the input / output tile in shared memory
constexpr int IMG_BYTES = 128 * 128;  // one weight image: [128 rows][64 k] bf16
constexpr int NCOMMON = 10;           // chunks every rank streams (pose encoder)
constexpr int NRANK = 6;              // packed [128][64] chunks per rank of the narrow head layout (kept in the blob)
constexpr int WIDE_BYTES = NHC * 128; // one wide head image: [192 n = this rank's 3 x 64 head columns][64 k] bf16, 24 KB
constexpr int ATOM_BYTES = 128 * 128; // A operand atom: [128 rows][64 k] bf16
constexpr uint32_t TMEM_COLS = 512;
constexpr int MAX_SLOTS = 5;          // objects a tile may span for the shared-memory proj table
constexpr uint32_t kIdescN128 = make_idesc_bf16(128, 128);
constexpr uint32_t kIdescN64 = make_idesc_bf16(128, 64);
constexpr uint32_t kIdescN192 = make_idesc_bf16(128, NHC);
constexpr uint32_t kIdescT128 = make_idesc_tf32(128, 128);
constexpr uint32_t kIdescT192 = make_idesc_tf32(128, NHC);
constexpr uint32_t COL_A_HI = 0, COL_A_LO = 128, COL_ACC = 256;   // TMEM columns: A operand (hi, lo), accumulators
static_assert(TrunkLayout::TC_CHUNKS == NCOMMON + CL * NRANK, "packed chunk count");
static_assert(TrunkLayout::WIDE_IMG_FLOATS * 4 == WIDE_BYTES, "wide head image size");

template <int NPASS>
struct Smem {
    static constexpr int IMAGES = NPASS == 1 ? 1 : 2;
    static constexpr int NSTAGE = NPASS == 1 ? 6 : 5;
    // one ring slot holds a pose-encoder chunk ([128][64] image; hi + lo in split mode, k 0..31 + k 32..63 in tf32
    // mode) or ONE wide head image (24 KB)
    static constexpr int SLOT = NPASS == 1 ? WIDE_BYTES : 2 * IMG_BYTES;
    // ring entries per evaluation: 10 pose-encoder chunks (all images of a chunk in one slot) + 4 k-atoms of the wide
    // head image (one slot per image)
    static constexpr int ENTRIES = NCOMMON + 4 * IMAGES;
    uint8_t ring[NSTAGE][SLOT];               // 160 / 144 KB; the struct sits on a 1024-byte boundary
    float stage[9 * RT];                      // this CTA's combined partial [c][row], source of the bulk copies to the peers
    float part[CL - 1][9 * RT];               // [peer][c][row] partial outputs, written by the other CTAs of the cluster;
                                              // compute_tq scratch between evaluations
    float4 wo[NHC];                           // output-layer weights of this rank's head columns
    float x[RT * XS];                         // inputs [RT][9]; overwritten with f_theta [RT][9] by forward()
    float pj[MAX_SLOTS * NHC];                // proj[obj][this rank's columns] for the objects of the tile
    float pjq[MAX_SLOTS * NHC];               // ... + this evaluation's t-branch (what the head epilogue adds to the accumulators)
    float tq[6 * NHC];                        // t-branch, up to 6 stages x this rank's columns
    float b1[256], b2[256];
    float bo[12];
    float times[8];
    double red[16];
    int obj[RT];
    unsigned long long full[NSTAGE], empty[NSTAGE], a_ready, dbar[5];
    unsigned long long stage_ready;   // this CTA's combined partial sits in the staging area (4 warp arrivals)
    unsigned long long xfull;         // the three peers' partials have landed in S.part (bulk-copy complete_tx)
    unsigned long long xfree;         // the three peers have consumed what this CTA sent them (remote arrivals)
    uint32_t tmem_base;
};

// pipeline state carried across evaluations (every thread holds a copy, each role uses its own fields)
struct State {
    uint32_t loads = 0;      // producer: chunks issued so far
    uint32_t consumed = 0;   // MMA issuer: chunks consumed so far
    uint32_t a_phase = 0;    // MMA issuer: parity of the next a_ready completion
    uint32_t d_phase = 0;    // epilogue: parity of this evaluation's dbar completions
    uint32_t rank = 0;       // cluster rank = which 64 columns of every head
    uint32_t evals = 0;      // evaluations done (parity of the exchange barriers)
    int tile_r0 = -1;        // tile whose obj / proj tables are loaded
    int slot_base = 0, nslots = 0;
    // cycle counters of one epilogue thread (phase breakdown of an evaluation, reported through `stats`)
    long long cyc_l1 = 0, cyc_wait1 = 0, cyc_epi1 = 0, cyc_waith = 0, cyc_epi2 = 0, cyc_fwd = 0;
    long long cyc_x[5] = {0, 0, 0, 0, 0};  // tail: combine halves, barrier A, scatter, barrier B, final sum
    long long cyc_wfull = 0;               // MMA issuer: cycles spent waiting for weight chunks (ring `full` barriers)
};

// global head column (0..767) of this rank's local column i (0..191)
__device__ __forceinline__ int head_col(uint32_t rank, int i) { return (i / HC) * 256 + HC * (int)rank + (i % HC); }

__device__ __forceinline__ const uint8_t *chunk_src(const float *__restrict__ P, uint32_t q, int which) {
    return reinterpret_cast<const uint8_t *>(P + TrunkLayout::W_TC) + ((size_t)q * 2 + which) * IMG_BYTES;
}

// entry L of the endless per-CTA stream: position i = L % ENTRIES inside an evaluation
template <int NPASS>
__device__ __forceinline__ void issue_chunk(Smem<NPASS> &S, const float *__restrict__ P, uint32_t L, uint32_t rank) {
    constexpr int NST = Smem<NPASS>::NSTAGE, IM = Smem<NPASS>::IMAGES, E = Smem<NPASS>::ENTRIES;
    const uint32_t s = L % NST, i = L % E;
    if (i < NCOMMON) {
        mbar_arrive_expect_tx(&S.full[s], IM * IMG_BYTES);
        for (int w = 0; w < IM; ++w) bulk_g2s(S.ring[s] + w * IMG_BYTES, chunk_src(P, i, w), IMG_BYTES, &S.full[s]);
    } else {
        // wide head image of this rank: k-atom kc, hi or lo ([192 n][64 k], TrunkLayout::W_WIDE)
        const uint32_t j = i - NCOMMON, kc = j / IM, which = j % IM;
        const uint8_t *src = reinterpret_cast<const uint8_t *>(P + TrunkLayout::W_WIDE) +
                             ((size_t)((rank * 4 + kc) * 2 + which)) * WIDE_BYTES;
        mbar_arrive_expect_tx(&S.full[s], WIDE_BYTES);
        bulk_g2s(S.ring[s], src, WIDE_BYTES, &S.full[s]);
    }
}

// one-time setup / teardown (all threads call)
template <int NPASS>
__device__ __forceinline__ void setup(Smem<NPASS> &S, State &st, const float *__restrict__ P) {
    constexpr int NST = Smem<NPASS>::NSTAGE;
    const int tid = threadIdx.x, warp = tid >> 5;
    st.rank = cluster_ctarank();
    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&S.full[s], 1); mbar_init(&S.empty[s], 1); }
        mbar_init(&S.a_ready, 8);
        for (int i = 0; i < 5; ++i) mbar_init(&S.dbar[i], 1);
        mbar_init(&S.stage_ready, 4);
        mbar_init(&S.xfull, 1);
        mbar_init(&S.xfree, CL - 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 256; i += NTHREADS) {
        S.b1[i] = __ldg(P + TrunkLayout::B1 + i);
        S.b2[i] = __ldg(P + TrunkLayout::B2 + i);
    }
    for (int i = tid; i < NHC; i += NTHREADS)
        S.wo[i] = __ldg(reinterpret_cast<const float4 *>(P + TrunkLayout::WO) + head_col(st.rank, i));
    if (tid < 12) S.bo[tid] = __ldg(P + TrunkLayout::BO + tid);
    __syncthreads();
    if (warp == 1) tmem_alloc(&S.tmem_base, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (tid == 0) {  // prefill the ring
        for (uint32_t L = 0; L < (uint32_t)NST; ++L) issue_chunk<NPASS>(S, P, L, st.rank);
        st.loads = NST;
    }
    __syncwarp();
    // every CTA of the cluster is running before anyone touches a peer's shared memory
    cluster_arrive();
    cluster_wait();
}

template <int NPASS>
__device__ __forceinline__ void teardown(Smem<NPASS> &S, State &st) {
    constexpr int NST = Smem<NPASS>::NSTAGE;
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 1 && (tid & 31) == 0) {  // drain the NSTAGE chunks that are still in flight
        for (int i = 0; i < NST; ++i) {
            const uint32_t g = st.consumed + i;
            mbar_wait(&S.full[g % NST], (g / NST) & 1);
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(S.tmem_base, TMEM_COLS);
    // no CTA leaves while a peer could still address its shared memory
    cluster_arrive();
    cluster_wait();
}

// byte offset of (row, column n) inside an A buffer (4 k-atoms of [128 rows][64 k] bf16, SWIZZLE_128B)
__device__ __forceinline__ int a_offset(int row, int n) {
    return (n >> 6) * ATOM_BYTES + row * 128 + ((((n & 63) >> 3) ^ (row & 7)) << 4) + ((n & 7) << 1);
}

// t-branch of `ns` stage times into S.tq[ns][NHC] (this rank's columns only); whole block; scratch = S.part
template <int NPASS>
__device__ __forceinline__ void compute_tq_rank(const float *__restrict__ P, Smem<NPASS> &S, const State &st, int ns) {
    const uint32_t rank = st.rank;
    static_assert(sizeof(S.part) >= 2048 * sizeof(float), "compute_tq scratch");
    compute_tq_cols(P, S.times, ns, &S.part[0][0], S.tq, NHC, [rank](int n) { return head_col(rank, n); });
}

// rows r0.. of the batch become the current tile: object of every row and the proj columns this rank needs.
// Callers synchronise the block (they fill S.x next) before forward().
template <int NPASS>
__device__ __forceinline__ void begin_tile(Smem<NPASS> &S, State &st, const float *__restrict__ proj, int r0, int N, int rpo) {
    if (st.tile_r0 == r0) return;
    st.tile_r0 = r0;
    const int tid = threadIdx.x;
    for (int r = tid; r < RT; r += NTHREADS) S.obj[r] = (r0 + r < N) ? (r0 + r) / rpo : -1;
    const int first = r0 / rpo, last = (min(r0 + RT, N) - 1) / rpo;
    st.slot_base = first;
    st.nslots = r0 < N ? last - first + 1 : 0;
    if (st.nslots <= MAX_SLOTS) {
        for (int i = tid; i < st.nslots * NHC; i += NTHREADS) {
            const int s = i / NHC, c = i - NHC * s;
            S.pj[i] = __ldg(proj + (size_t)(first + s) * 768 + head_col(st.rank, c));
        }
    }
}

// TMEM accumulator columns [dcol + c0, dcol + c0 + 128) of this thread's row -> relu(. + bias) -> bf16 (hi / lo)
// -> A operand buffers
template <int NPASS>
__device__ __forceinline__ void epi_hidden(uint32_t taddr, const float *sbias, int row, int c0, uint32_t A_hi, uint32_t A_lo) {
    // two register buffers: the TMEM load of the next 32 columns is in flight while these are converted
    // (tcgen05.ld is scoreboarded in hardware; the formal wait::ld before the first use compiles to nothing)
    uint32_t r[2][32];
    tmem_ld32_nowait(taddr + c0, r[0]);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        if (g + 1 < 4) tmem_ld32_nowait(taddr + c0 + (g + 1) * 32, r[(g + 1) & 1]);
        tmem_ld_wait();
#pragma unroll
        for (int j8 = 0; j8 < 4; ++j8) {
            const int n0 = c0 + g * 32 + j8 * 8;
            float v[8];
            const float4 ba = *reinterpret_cast<const float4 *>(sbias + n0), bb = *reinterpret_cast<const float4 *>(sbias + n0 + 4);
            const float bv[8] = {ba.x, ba.y, ba.z, ba.w, bb.x, bb.y, bb.z, bb.w};
#pragma unroll
            for (int j = 0; j < 8; ++j) v[j] = fmaxf(__uint_as_float(r[g & 1][j8 * 8 + j]) + bv[j], 0.f);
            const __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
            const __nv_bfloat162 p2 = __floats2bfloat162_rn(v[4], v[5]), p3 = __floats2bfloat162_rn(v[6], v[7]);
            uint4 pk;
            pk.x = *reinterpret_cast<const uint32_t *>(&p0); pk.y = *reinterpret_cast<const uint32_t *>(&p1);
            pk.z = *reinterpret_cast<const uint32_t *>(&p2); pk.w = *reinterpret_cast<const uint32_t *>(&p3);
            const int off = a_offset(row, n0);
            sts_u4(A_hi + off, pk);
            if (NPASS == 3) {
                const float2 f0 = __bfloat1622float2(p0), f1 = __bfloat1622float2(p1);
                const float2 f2 = __bfloat1622float2(p2), f3 = __bfloat1622float2(p3);
                const __nv_bfloat162 l0 = __floats2bfloat162_rn(v[0] - f0.x, v[1] - f0.y), l1 = __floats2bfloat162_rn(v[2] - f1.x, v[3] - f1.y);
                const __nv_bfloat162 l2 = __floats2bfloat162_rn(v[4] - f2.x, v[5] - f2.y), l3 = __floats2bfloat162_rn(v[6] - f3.x, v[7] - f3.y);
                uint4 pl;
                pl.x = *reinterpret_cast<const uint32_t *>(&l0); pl.y = *reinterpret_cast<const uint32_t *>(&l1);
                pl.z = *reinterpret_cast<const uint32_t *>(&l2); pl.w = *reinterpret_cast<const uint32_t *>(&l3);
                sts_u4(A_lo + off, pl);
            }
        }
    }
}

// accumulator columns [acc + c0, acc + c0 + 128) of this thread's row -> relu(. + bias) -> packed bf16 (hi / lo)
// -> the A operand in TMEM (k = output column: 32 output columns = 16 packed 32-bit columns)
// (tf32 mode: 32 output columns = 32 TMEM columns of tf32-rounded values)
template <int NPASS>
__device__ __forceinline__ void epi_hidden_t(uint32_t lane_addr, uint32_t acc, const float *sbias, int c0) {
    uint32_t r[2][32];
    if constexpr (NPASS == 2) {
        tmem_ld32_nowait(lane_addr + acc + c0, r[0]);
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            if (g + 1 < 4) tmem_ld32_nowait(lane_addr + acc + c0 + (g + 1) * 32, r[(g + 1) & 1]);
            tmem_ld_wait();
            uint32_t v[2][16];
#pragma unroll
            for (int j4 = 0; j4 < 8; ++j4) {
                const float4 b = *reinterpret_cast<const float4 *>(sbias + c0 + g * 32 + j4 * 4);
                const float bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    v[j4 >> 2][(j4 & 3) * 4 + j] = __float_as_uint(tf32_rna(fmaxf(__uint_as_float(r[g & 1][j4 * 4 + j]) + bv[j], 0.f)));
            }
            const uint32_t kcol = (uint32_t)(c0 + g * 32);
            tmem_st16(lane_addr + COL_A_HI + kcol, v[0]);
            tmem_st16(lane_addr + COL_A_HI + kcol + 16, v[1]);
        }
        tmem_st_wait();
        return;
    }
    tmem_ld32_nowait(lane_addr + acc + c0, r[0]);
#pragma unroll
    for (int g = 0; g < 4; ++g) {
        if (g + 1 < 4) tmem_ld32_nowait(lane_addr + acc + c0 + (g + 1) * 32, r[(g + 1) & 1]);
        tmem_ld_wait();
        uint32_t hi[16], lo[16];
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
            const int n0 = c0 + g * 32 + j4 * 4;
            const float4 b = *reinterpret_cast<const float4 *>(sbias + n0);
            const float v0 = fmaxf(__uint_as_float(r[g & 1][j4 * 4 + 0]) + b.x, 0.f), v1 = fmaxf(__uint_as_float(r[g & 1][j4 * 4 + 1]) + b.y, 0.f);
            const float v2 = fmaxf(__uint_as_float(r[g & 1][j4 * 4 + 2]) + b.z, 0.f), v3 = fmaxf(__uint_as_float(r[g & 1][j4 * 4 + 3]) + b.w, 0.f);
            const __nv_bfloat162 p0 = __floats2bfloat162_rn(v0, v1), p1 = __floats2bfloat162_rn(v2, v3);
            hi[j4 * 2 + 0] = *reinterpret_cast<const uint32_t *>(&p0);
            hi[j4 * 2 + 1] = *reinterpret_cast<const uint32_t *>(&p1);
            if (NPASS == 3) {
                const float2 f0 = __bfloat1622float2(p0), f1 = __bfloat1622float2(p1);
                const __nv_bfloat162 l0 = __floats2bfloat162_rn(v0 - f0.x, v1 - f0.y), l1 = __floats2bfloat162_rn(v2 - f1.x, v3 - f1.y);
                lo[j4 * 2 + 0] = *reinterpret_cast<const uint32_t *>(&l0);
                lo[j4 * 2 + 1] = *reinterpret_cast<const uint32_t *>(&l1);
            }
        }
        const uint32_t kcol = (uint32_t)(c0 + g * 32) >> 1;
        tmem_st16(lane_addr + COL_A_HI + kcol, hi);
        if (NPASS == 3) tmem_st16(lane_addr + COL_A_LO + kcol, lo);
    }
    tmem_st_wait();
}

// inputs (k 0..8, k 9..15 zero) of this thread's row -> the A operand in TMEM: 8 packed bf16 columns (hi, and lo in
// split mode) or 16 tf32 columns
template <int NPASS>
__device__ __forceinline__ void store_x_bf16(uint32_t lane_addr, const float (&xv)[9]) {
    uint32_t hi[8], lo[8];
#pragma unroll
    for (int p = 0; p < 8; ++p) {
        const float v0 = 2 * p < 9 ? xv[2 * p] : 0.f, v1 = 2 * p + 1 < 9 ? xv[2 * p + 1] : 0.f;
        const __nv_bfloat162 h2 = __floats2bfloat162_rn(v0, v1);
        const float2 hf = __bfloat1622float2(h2);
        const __nv_bfloat162 l2 = __floats2bfloat162_rn(v0 - hf.x, v1 - hf.y);
        hi[p] = *reinterpret_cast<const uint32_t *>(&h2);
        lo[p] = *reinterpret_cast<const uint32_t *>(&l2);
    }
    tmem_st8(lane_addr + COL_A_HI, hi);
    if (NPASS == 3) tmem_st8(lane_addr + COL_A_LO, lo);
}
__device__ __forceinline__ void store_x_tf32(uint32_t lane_addr, const float (&xv)[9]) {
    uint32_t v[16];
#pragma unroll
    for (int k = 0; k < 16; ++k) v[k] = k < 9 ? __float_as_uint(tf32_rna(xv[k])) : 0u;
    tmem_st16(lane_addr + COL_A_HI, v);
}

// Head epilogue of one head for a warp's 32 rows x 32 accumulator columns: z = relu(D + e) and the 256 -> 3 output layer over
// these columns.  The accumulators are read in the 16x256b fragment layout: a thread holds 8 columns (8 i + 2 (lane & 3) + {0, 1})
// of 4 rows (TMEM lanes (lane >> 2) + 8 k of the warp's quarter), so an output-layer weight is loaded once per 4 rows -- with
// one row per thread (32x32b) the broadcast LDS.128 per column (512 B of register write-back each) bound the epilogue.
// The 4 lanes that share rows then reduce-scatter their partial sums: thread (lane) ends up with the 3 outputs of ONE row,
// TMEM lane (lane >> 2) + 8 (lane & 3).  e_k: the row's proj + tq columns (shared-memory table, or global proj + tq when TABLE
// is false).  Split into load / compute / reduce so that the TMEM load of the next block is in flight under the FMAs of this one.
struct HeadFrag {
    uint32_t ra[16], rb[16];   // rows k = 0, 1 (TMEM lanes + 0..15 of the quarter) and k = 2, 3 (lanes + 16..31)
};
// request a 32-row x 32-column accumulator block of the warp's quarter (no wait: tmem_ld_wait() before head_compute)
__device__ __forceinline__ void head_load(uint32_t quarter_addr, uint32_t col, HeadFrag &f) {
    tmem_ld_16x256b_x4_nowait(quarter_addr + col, f.ra);
    tmem_ld_16x256b_x4_nowait(quarter_addr + (16u << 16) + col, f.rb);
}
// a[k][o] += sum over this thread's 8 columns of relu(D[row k][c] + e_k[c]) * Wo[c][o]
template <bool TABLE>
__device__ __forceinline__ void head_compute(const HeadFrag &f, const float4 *swo_cb, const float *const (&erow)[4],
                                             const float *stq_cb, int lane, float (&a)[4][3]) {
    const int tq4 = lane & 3;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int cc = 8 * i + 2 * tq4;
        const float4 w0 = swo_cb[cc], w1 = swo_cb[cc + 1];
        float2 tqv = make_float2(0.f, 0.f);
        if (!TABLE) tqv = *reinterpret_cast<const float2 *>(stq_cb + cc);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            float2 e;
            if (TABLE) {
                e = *reinterpret_cast<const float2 *>(erow[k] + cc);
            } else {
                const float2 g = __ldg(reinterpret_cast<const float2 *>(erow[k] + cc));
                e = make_float2(g.x + tqv.x, g.y + tqv.y);
            }
            const uint32_t d0 = k < 2 ? f.ra[4 * i + 2 * (k & 1)] : f.rb[4 * i + 2 * (k & 1)];
            const uint32_t d1 = k < 2 ? f.ra[4 * i + 2 * (k & 1) + 1] : f.rb[4 * i + 2 * (k & 1) + 1];
            const float z0 = fmaxf(__uint_as_float(d0) + e.x, 0.f), z1 = fmaxf(__uint_as_float(d1) + e.y, 0.f);
            a[k][0] = fmaf(z1, w1.x, fmaf(z0, w0.x, a[k][0]));
            a[k][1] = fmaf(z1, w1.y, fmaf(z0, w0.y, a[k][1]));
            a[k][2] = fmaf(z1, w1.z, fmaf(z0, w0.z, a[k][2]));
        }
    }
}
// reduce-scatter over the 4 lanes of a row group (xor 2 halves the rows a lane keeps, xor 1 again): out = the 3 sums of
// row k = lane & 3
__device__ __forceinline__ void head_reduce(const float (&a)[4][3], int lane, float (&out)[3]) {
    const bool up2 = (lane & 2) != 0, up1 = (lane & 1) != 0;
#pragma unroll
    for (int o = 0; o < 3; ++o) {
        const float s0 = up2 ? a[0][o] : a[2][o], s1 = up2 ? a[1][o] : a[3][o];
        float k0 = up2 ? a[2][o] : a[0][o], k1 = up2 ? a[3][o] : a[1][o];
        k0 += __shfl_xor_sync(0xffffffffu, s0, 2);
        k1 += __shfl_xor_sync(0xffffffffu, s1, 2);
        const float s = up1 ? k0 : k1, kk = up1 ? k1 : k0;
        out[o] = kk + __shfl_xor_sync(0xffffffffu, s, 1);
    }
}

// f_theta for the 128 rows in S.x -> S.x [r*9 + c]; `tq` is this stage's t-branch (NHC floats in shared memory,
// this rank's columns).  All 320 threads of all CL CTAs of the cluster call; ends with __syncthreads().
template <int NPASS>
__device__ __noinline__ void forward(const float *__restrict__ P, const float *__restrict__ proj, Smem<NPASS> &S,
                                     State &st, const float *tq) {
    constexpr int NST = Smem<NPASS>::NSTAGE;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t tmem = S.tmem_base;
    const uint32_t rank = st.rank;
    const long long t_begin = clock64();
    long long tx = 0;
    float acc[9];   // epilogue threads: this row's partial output over the thread's columns

    const uint32_t xph = st.evals & 1;

    if (warp == 0) {
        // ---------------- TMA producer ----------------
        if (lane == 0) {
            mbar_arrive_expect_tx(&S.xfull, (CL - 1) * 9 * RT * sizeof(float));  // this evaluation's incoming partials
            for (int i = 0; i < Smem<NPASS>::ENTRIES; ++i) {
                const uint32_t L = st.loads;
                mbar_wait(&S.empty[L % NST], ((L / NST) + 1) & 1);
                issue_chunk<NPASS>(S, P, L, rank);
                st.loads = L + 1;
            }
            // exchange: once the combined partial of this CTA is staged and the peers have consumed the previous
            // one, copy it into their S.part slot (async proxy, completes on their xfull: no thread fences)
            mbar_wait(&S.stage_ready, xph);
            if (st.evals > 0) mbar_wait(&S.xfree, xph ^ 1);
            const float *stage = S.stage;
            for (uint32_t d = 0; d < (uint32_t)CL; ++d) {
                if (d == rank) continue;
                bulk_s2peer(mapa(smem_u32(&S.part[rank < d ? rank : rank - 1][0]), d), stage, 9 * RT * sizeof(float),
                            mapa(smem_u32(&S.xfull), d));
            }
            bulk_wait_read();  // the staging area is free again when forward() returns
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---------------- MMA issuer ----------------
        if (lane == 0) {
            const uint32_t a_hi = tmem + COL_A_HI, a_lo = tmem + COL_A_LO, acc = tmem + COL_ACC;
            uint32_t b_hi = 0, b_lo = 0, stage = 0;
            auto next_chunk = [&]() {
                const uint32_t g = st.consumed;
                stage = g % NST;
                const long long w0 = clock64();
                mbar_wait(&S.full[stage], (g / NST) & 1);
                st.cyc_wfull += clock64() - w0;
                tc_fence_after();
                b_hi = smem_u32(&S.ring[stage][0]);
                b_lo = b_hi + (NPASS != 1 ? IMG_BYTES : 0);
            };
            auto chunk_done = [&]() {
                umma_commit(&S.empty[stage]);
                st.consumed += 1;
            };
            // the 1 / 3 products of one k step (A columns `ac`: 8 packed TMEM columns = 16 k) against the chunk's B images
            auto mma = [&](uint32_t d, uint32_t ac, uint32_t bo, uint32_t idesc, uint32_t accum) {
                umma_bf16_ts(d, a_hi + ac, make_desc(b_hi + bo), idesc, accum);
                if (NPASS == 3) {
                    umma_bf16_ts(d, a_lo + ac, make_desc(b_hi + bo), idesc, 1u);
                    umma_bf16_ts(d, a_hi + ac, make_desc(b_lo + bo), idesc, 1u);
                }
            };
            // pose_encoder.0: K = 16 (9 used), D0 -> accumulator cols 0..255
            mbar_wait(&S.a_ready, st.a_phase); st.a_phase ^= 1;
            tc_fence_after();
            for (int nh = 0; nh < 2; ++nh) {
                next_chunk();
                if constexpr (NPASS == 2) {   // k 0..7, 8..15 of the first image
                    umma_tf32_ts(acc + nh * 128, a_hi, make_desc(b_hi), kIdescT128, 0u);
                    umma_tf32_ts(acc + nh * 128, a_hi + 8, make_desc(b_hi + 32), kIdescT128, 1u);
                } else {
                    mma(acc + nh * 128, 0, 0, kIdescN128, 0u);
                }
                chunk_done();
            }
            umma_commit(&S.dbar[0]);
            // pose_encoder.2: D1 -> the same accumulator columns (D0 has been read out).  Consecutive MMAs into one
            // accumulator form a dependent chain (~90 cycles each, an N128 MMA occupies the pipe for 64): the two column
            // halves of a k-atom are multiplied interleaved, two independent accumulators in flight.
            mbar_wait(&S.a_ready, st.a_phase); st.a_phase ^= 1;
            tc_fence_after();
            for (int kc = 0; kc < 4; ++kc) {
                const uint32_t g = st.consumed, s0 = g % NST, s1 = (g + 1) % NST;
                const long long w0 = clock64();
                mbar_wait(&S.full[s0], (g / NST) & 1);
                mbar_wait(&S.full[s1], ((g + 1) / NST) & 1);
                st.cyc_wfull += clock64() - w0;
                tc_fence_after();
                const uint32_t b0 = smem_u32(&S.ring[s0][0]), b1 = smem_u32(&S.ring[s1][0]);
                const uint32_t bl0 = b0 + (NPASS == 3 ? IMG_BYTES : 0), bl1 = b1 + (NPASS == 3 ? IMG_BYTES : 0);
                if constexpr (NPASS == 2) {
#pragma unroll
                    for (int k8 = 0; k8 < 8; ++k8) {   // image k8 / 4 of the chunk, A columns = k
                        const uint32_t ac = kc * 64 + k8 * 8, bo = (k8 >> 2) * IMG_BYTES + (k8 & 3) * 32;
                        const uint32_t accum = (kc | k8) ? 1u : 0u;
                        umma_tf32_ts(acc, a_hi + ac, make_desc(b0 + bo), kIdescT128, accum);
                        umma_tf32_ts(acc + 128, a_hi + ac, make_desc(b1 + bo), kIdescT128, accum);
                    }
                } else {
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk) {
                        const uint32_t ac = kc * 32 + kk * 8, bo = kk * 32, accum = (kc | kk) ? 1u : 0u;
                        umma_bf16_ts(acc, a_hi + ac, make_desc(b0 + bo), kIdescN128, accum);
                        umma_bf16_ts(acc + 128, a_hi + ac, make_desc(b1 + bo), kIdescN128, accum);
                        if (NPASS == 3) {
                            umma_bf16_ts(acc, a_lo + ac, make_desc(b0 + bo), kIdescN128, 1u);
                            umma_bf16_ts(acc + 128, a_lo + ac, make_desc(b1 + bo), kIdescN128, 1u);
                            umma_bf16_ts(acc, a_hi + ac, make_desc(bl0 + bo), kIdescN128, 1u);
                            umma_bf16_ts(acc + 128, a_hi + ac, make_desc(bl1 + bo), kIdescN128, 1u);
                        }
                    }
                }
                umma_commit(&S.empty[s0]);
                umma_commit(&S.empty[s1]);
                st.consumed = g + 2;
            }
            umma_commit(&S.dbar[1]);
            // heads: this rank's 64 columns of each head as ONE N = 192 accumulator, accumulator cols 0..191 (D1 has
            // been read out): the A operand (h2) is read once per k step for all three heads, and an N = 192 MMA occupies
            // the pipe for 96 cycles >= the accumulate latency, so one chain keeps the pipe busy.
            // Column 64 h + c of the accumulator = head h, column 64 rank + c.
            mbar_wait(&S.a_ready, st.a_phase); st.a_phase ^= 1;
            tc_fence_after();
            for (int kc = 0; kc < 4; ++kc) {
                if constexpr (NPASS == 2) {
                    for (int w = 0; w < 2; ++w) {   // k 0..31, then k 32..63 of the k-atom
                        next_chunk();
#pragma unroll
                        for (int kk = 0; kk < 4; ++kk)
                            umma_tf32_ts(acc, a_hi + kc * 64 + w * 32 + kk * 8, make_desc(b_hi + kk * 32), kIdescT192,
                                         (kc | w | kk) ? 1u : 0u);
                        chunk_done();
                    }
                    continue;
                }
                next_chunk();   // hi image
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {
                    const uint32_t ac = kc * 32 + kk * 8;
                    umma_bf16_ts(acc, a_hi + ac, make_desc(b_hi + kk * 32), kIdescN192, (kc | kk) ? 1u : 0u);
                    if (NPASS == 3) umma_bf16_ts(acc, a_lo + ac, make_desc(b_hi + kk * 32), kIdescN192, 1u);
                }
                chunk_done();
                if (NPASS == 3) {
                    next_chunk();   // lo image
#pragma unroll
                    for (int kk = 0; kk < 4; ++kk)
                        umma_bf16_ts(acc, a_hi + kc * 32 + kk * 8, make_desc(b_hi + kk * 32), kIdescN192, 1u);
                    chunk_done();
                }
            }
            umma_commit(&S.dbar[2]);
            umma_commit(&S.dbar[3]);
            umma_commit(&S.dbar[4]);
        }
        __syncwarp();
    } else {
        // ---------------- epilogue warps ----------------
        const int e = warp - 2;
        const int row = 32 * (warp & 3) + lane;   // TMEM lane quarter is fixed by warp % 4
        const int half = e >> 2;                  // column half 0 / 1
        const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
        const uint32_t dph = st.d_phase;
        st.d_phase ^= 1;
        // Views derived from the dynamic shared array itself: the compiler then knows the address space (LDS,
        // freely schedulable) although S is only reachable through a generic pointer.
        extern __shared__ __align__(16) unsigned char gp_dyn_smem[];
        const uint32_t dyn0 = smem_u32(gp_dyn_smem);
        const float *sx = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.x) - dyn0));
        const float *sb1 = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.b1) - dyn0));
        const float *sb2 = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.b2) - dyn0));
        const float *spj = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.pj) - dyn0));
        float *spjq = reinterpret_cast<float *>(gp_dyn_smem + (smem_u32(S.pjq) - dyn0));
        const float *stq = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(tq) - dyn0));
        const float4 *swo = reinterpret_cast<const float4 *>(gp_dyn_smem + (smem_u32(S.wo) - dyn0));
        float *sxw = reinterpret_cast<float *>(gp_dyn_smem + (smem_u32(S.x) - dyn0));

        long long t0 = clock64();
        // inputs -> A operand: k 0..8 of atom 0 (k 9..15 zero), one row per thread of the first four warps
        if (half == 0) {
            float xv[9];
#pragma unroll
            for (int c = 0; c < 9; ++c) xv[c] = sx[row * XS + c];
            if constexpr (NPASS == 2) store_x_tf32(lane_addr, xv);
            else store_x_bf16<NPASS>(lane_addr, xv);
            tmem_st_wait();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.a_ready);
        // while the first layer runs: proj + this stage's t-branch for the objects of the tile (consumed by the head epilogue
        // after the named barrier below)
        const bool use_pj = st.nslots <= MAX_SLOTS;
        if (use_pj)
            for (int i = tid - 64; i < st.nslots * NHC; i += 256) spjq[i] = spj[i] + stq[i % NHC];

        // h1 = relu(D0 + b1) -> A buffers
        mbar_wait(&S.dbar[0], dph);
        tc_fence_after();
        epi_hidden_t<NPASS>(lane_addr, COL_ACC, sb1, half * 128);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.a_ready);
        {
            const long long t1 = clock64();
            st.cyc_l1 += t1 - t0;
            t0 = t1;
        }
        // h2 = relu(D1 + b2) -> A buffers
        mbar_wait(&S.dbar[1], dph);
        tc_fence_after();
        {
            const long long t1 = clock64();
            st.cyc_wait1 += t1 - t0;
            t0 = t1;
        }
        epi_hidden_t<NPASS>(lane_addr, COL_ACC, sb2, half * 128);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.a_ready);
        {
            const long long t1 = clock64();
            st.cyc_epi1 += t1 - t0;
            t0 = t1;
        }

        // heads: z = relu(D + proj + tq), partial out = z . Wo^T over this warp's 32 columns of each head (head_block)
        asm volatile("bar.sync 3, 256;" ::: "memory");   // S.pjq is complete (the 8 epilogue warps)
        const int tq4 = lane & 3, tr = lane >> 2;
        const int q32 = 32 * (warp & 3);
        const float *erow[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int o = S.obj[q32 + tr + 8 * k];
            erow[k] = use_pj ? spjq + (o >= 0 ? o - st.slot_base : 0) * NHC : proj + (size_t)(o < 0 ? 0 : o) * 768;
        }
        float out9[9];
        // the three heads complete together (one commit): request head h + 1 while head h is multiplied
        mbar_wait(&S.dbar[2], dph);
        mbar_wait(&S.dbar[3], dph);
        mbar_wait(&S.dbar[4], dph);
        tc_fence_after();
        {
            const long long t1 = clock64();
            st.cyc_waith += t1 - t0;
            t0 = t1;
        }
        HeadFrag frag[2];
        head_load(lane_addr, COL_ACC + half * 32, frag[0]);
#pragma unroll
        for (int h = 0; h < 3; ++h) {
            tmem_ld_wait();
            if (h + 1 < 3) head_load(lane_addr, COL_ACC + (h + 1) * HC + half * 32, frag[(h + 1) & 1]);
            const int cb = h * HC + half * 32;                      // local column base
            const int gcol = h * 256 + HC * (int)rank + half * 32;  // global head column base
            const float *e4[4];
#pragma unroll
            for (int k = 0; k < 4; ++k) e4[k] = erow[k] + (use_pj ? cb : gcol);
            float a[4][3];
#pragma unroll
            for (int k = 0; k < 4; ++k) a[k][0] = a[k][1] = a[k][2] = 0.f;
            if (use_pj) head_compute<true>(frag[h & 1], swo + cb, e4, stq + cb, lane, a);
            else head_compute<false>(frag[h & 1], swo + cb, e4, stq + cb, lane, a);
            float o3[3];
            head_reduce(a, lane, o3);
            out9[h * 3 + 0] = o3[0]; out9[h * 3 + 1] = o3[1]; out9[h * 3 + 2] = o3[2];
        }
        {
            const long long t1 = clock64();
            st.cyc_epi2 += t1 - t0;
            t0 = t1;
        }
        tc_fence_before();
        tx = clock64();
        // the two column halves of a row meet through shared memory: this thread holds the partial of row q32 + tr + 8 tq4;
        // half 0 parks it in the staging area (free: the previous evaluation's copies have read it), half 1 in S.x (dead since
        // the inputs were converted); then the row's owner thread of half 0 adds the two
        float *stage_w = reinterpret_cast<float *>(gp_dyn_smem + (smem_u32(S.stage) - dyn0));
        {
            float *dst = half ? sxw : stage_w;
            const int prow_l = q32 + tr + 8 * tq4;
#pragma unroll
            for (int c = 0; c < 9; ++c) dst[c * RT + prow_l] = out9[c];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");  // the 8 epilogue warps only
        if (half == 0) {
#pragma unroll
            for (int c = 0; c < 9; ++c) acc[c] = stage_w[c * RT + row] + sxw[c * RT + row];
        }
        { const long long t1 = clock64(); st.cyc_x[0] += t1 - tx; tx = t1; }
        if (half == 0) {
            // stage the row's partial [c][row] for the producer thread's bulk copies
            float *stage = reinterpret_cast<float *>(gp_dyn_smem + (smem_u32(S.stage) - dyn0));
#pragma unroll
            for (int c = 0; c < 9; ++c) stage[c * RT + row] = acc[c];
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(&S.stage_ready);
            { const long long t1 = clock64(); st.cyc_x[2] += t1 - tx; tx = t1; }
            // the peers' partials; every CTA adds the four in rank order: bit-identical f_theta in the whole cluster
            mbar_wait(&S.xfull, xph);
            // S.x turns from scratch into the output tile: every half-0 warp is past its scratch reads
            asm volatile("bar.sync 2, 128;" ::: "memory");
            { const long long t1 = clock64(); st.cyc_x[3] += t1 - tx; tx = t1; }
            const float *spart = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(&S.part[0][0]) - dyn0));
            const float *sbo = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.bo) - dyn0));
#pragma unroll
            for (int c = 0; c < 9; ++c) {
                float p[CL];
#pragma unroll
                for (uint32_t s = 0; s < (uint32_t)CL; ++s)
                    p[s] = s == rank ? acc[c] : spart[(s < rank ? s : s - 1) * 9 * RT + c * RT + row];
                sxw[row * XS + c] = ((p[0] + p[1]) + (p[2] + p[3])) + sbo[c];
            }
        }
    }
    __syncthreads();
    // credit: this CTA has consumed the partials it received
    if (tid == 32) {
        for (uint32_t d = 0; d < (uint32_t)CL; ++d)
            if (d != rank) mbar_arrive_peer_relaxed(mapa(smem_u32(&S.xfree), d));
    }
    st.evals += 1;
    st.cyc_x[4] += clock64() - tx;
    st.cyc_fwd += clock64() - t_begin;
}

}  // namespace tc
}  // namespace gp
