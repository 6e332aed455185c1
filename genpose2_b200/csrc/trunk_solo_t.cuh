// One-CTA-per-tile tensor-core evaluator of the ScoreNet trunk with the A OPERAND IN TENSOR MEMORY.
//
// Same decomposition as trunk_solo.cuh (one CTA per 128-row tile, no redundant work, one copy of the state), but the
// activations x / h1 / h2 never go through shared memory: the epilogue warps write them as packed bf16 pairs straight
// into TMEM (tcgen05.st) and the MMAs read their A operand from there (tcgen05.mma [d], [a_tmem], b_desc).  That
//   * removes the A-operand reads from the shared-memory pipe (an M128 x N128 x K16 MMA with both operands in shared
//     memory reads 8 KB for 64 cycles of math -- exactly the 128 B/clk the pipe delivers, so any other traffic stalls it);
//   * removes the swizzled st.shared + fence.proxy.async of the epilogues;
//   * frees the 64 / 128 KB A buffer: the weight ring becomes 8 x 16 KB deep, so the weight stream (L2 -> shared memory,
//     ~1.3 k cycles round trip per image) is no longer limited by two or three images in flight.
//
// TMEM map (512 columns x 128 lanes, lane = row of the tile):
//   [  0..127]  A hi : 256 k as packed bf16 pairs (column j = k 2j, 2j+1)      [128..255]  A lo (split mode)
//   (tf32 mode: [0..255] = 256 k, column k = tf32 value of k; a weight chunk's two images hold k 0..31 and 32..63)
//   [256..383]  accumulator slot 0                                            [384..511]  accumulator slot 1
// Per evaluation:
//   x (K = 16)  -> D0 = slots 0|1 (N = 256)  -> h1 = relu(D0 + b1) -> A
//   h1          -> D1 = slots 0|1            -> h2 = relu(D1 + b2) -> A (in place: D1 is complete before h2 is written)
//   h2          -> six half-heads (head h, columns 128 nh .. 128 nh + 127), alternating between the two slots: the
//                  epilogue of half-head i (+ proj + tq, ReLU, 256 -> 3 output layer) runs under the MMAs of i + 1.
#pragma once
#include "trunk_solo.cuh"

namespace gp {
namespace solot {

using namespace tc;

constexpr int NCHUNKS = 34;          // 2 (pose_encoder.0) + 8 (pose_encoder.2) + 3 x 8 (heads)
constexpr int SLOTS = 4;             // objects a tile may span for the shared-memory proj table
constexpr int NSTAGE = 8;            // ring depth (single 16 KB images)
// TMEM columns COL_A_HI / COL_A_LO / COL_ACC and epi_hidden_t come from trunk_tc.cuh (shared with the cluster shape)

template <int NPASS>
struct Smem {
    static constexpr int IMAGES = NPASS == 1 ? 1 : 2;
    static constexpr int ENTRIES = NCHUNKS * IMAGES;   // ring entries (single images) per evaluation
    uint8_t ring[NSTAGE][IMG_BYTES];          // 128 KB; the struct sits on a 1024-byte boundary
    float4 wo[768];                           // output-layer weights per head column (3 used)
    float tq[6 * 768];                        // t-branch, up to 6 stages
    float pj[SLOTS * 768];                    // proj rows of the objects of the tile
    float scratch[2048];                      // compute_tq scratch; the two column halves of a row meet here
    float x[RT * XS];                         // inputs [RT][9]; overwritten with f_theta [RT][9] by forward()
    float b1[256], b2[256];
    float bo[12];
    float times[8];
    double red[16];
    unsigned long long full[NSTAGE], empty[NSTAGE], a_ready, dbar[2], hbar[6], drain[4];
    uint32_t tmem_base;
};

struct State {
    uint32_t loads = 0;      // producer: ring entries issued so far
    uint32_t consumed = 0;   // MMA issuer: ring entries consumed so far
    uint32_t a_phase = 0;    // MMA issuer: parity of the next a_ready completion
    uint32_t evals = 0;      // evaluations done (parity of the once-per-evaluation barriers)
    int tile_r0 = -1;        // tile whose proj table is loaded
    int slot_base = 0, nslots = 0, rpo = 1, nrows = 0;
    long long cyc_fwd = 0, cyc_l1 = 0, cyc_wait1 = 0, cyc_epi1 = 0, cyc_waith = 0, cyc_epi2 = 0, cyc_tail = 0;
};

// ring entry L of the endless per-CTA stream -> source image.  Order inside an evaluation: pose_encoder.0 (n-half 0, 1),
// pose_encoder.2 (k-atom major, n-half inner), then per half-head (head h, n-half nh) its four k-atoms; hi then lo image.
template <int NPASS>
__device__ __forceinline__ const uint8_t *entry_src(const float *__restrict__ P, uint32_t L) {
    constexpr int IM = Smem<NPASS>::IMAGES;
    const uint32_t e = L % (uint32_t)Smem<NPASS>::ENTRIES;
    const uint32_t c = e / IM, which = e % IM;
    const uint8_t *base;
    if (c < 10) {
        base = reinterpret_cast<const uint8_t *>(P + TrunkLayout::W_TC) + (size_t)c * 2 * IMG_BYTES;
    } else {
        const uint32_t j = c - 10, h = j / 8, nh = (j % 8) / 4, kc = j % 4;
        base = reinterpret_cast<const uint8_t *>(P + TrunkLayout::W_SOLO) + (size_t)(8 * h + 2 * kc + nh) * 2 * IMG_BYTES;
    }
    return base + (size_t)which * IMG_BYTES;
}

template <int NPASS>
__device__ __forceinline__ void issue_entry(Smem<NPASS> &S, const float *__restrict__ P, uint32_t L) {
    const uint32_t s = L % (uint32_t)NSTAGE;
    mbar_arrive_expect_tx(&S.full[s], IMG_BYTES);
    bulk_g2s(S.ring[s], entry_src<NPASS>(P, L), IMG_BYTES, &S.full[s]);
}

template <int NPASS>
__device__ __forceinline__ void setup(Smem<NPASS> &S, State &st, const float *__restrict__ P) {
    const int tid = threadIdx.x, warp = tid >> 5;
    if (tid == 0) {
        for (int s = 0; s < NSTAGE; ++s) { mbar_init(&S.full[s], 1); mbar_init(&S.empty[s], 1); }
        mbar_init(&S.a_ready, 8);
        for (int i = 0; i < 2; ++i) mbar_init(&S.dbar[i], 1);
        for (int i = 0; i < 6; ++i) mbar_init(&S.hbar[i], 1);
        for (int i = 0; i < 4; ++i) mbar_init(&S.drain[i], 8);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 256; i += NTHREADS) {
        S.b1[i] = __ldg(P + TrunkLayout::B1 + i);
        S.b2[i] = __ldg(P + TrunkLayout::B2 + i);
    }
    for (int i = tid; i < 768; i += NTHREADS) S.wo[i] = __ldg(reinterpret_cast<const float4 *>(P + TrunkLayout::WO) + i);
    if (tid < 12) S.bo[tid] = __ldg(P + TrunkLayout::BO + tid);
    __syncthreads();
    if (warp == 1) tmem_alloc(&S.tmem_base, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    if (tid == 0) {  // prefill the ring
        for (uint32_t L = 0; L < (uint32_t)NSTAGE; ++L) issue_entry<NPASS>(S, P, L);
        st.loads = NSTAGE;
    }
    __syncwarp();
}

template <int NPASS>
__device__ __forceinline__ void teardown(Smem<NPASS> &S, State &st) {
    const int tid = threadIdx.x, warp = tid >> 5;
    if (warp == 1 && (tid & 31) == 0) {  // drain the entries that are still in flight
        for (int i = 0; i < NSTAGE; ++i) {
            const uint32_t g = st.consumed + i;
            mbar_wait(&S.full[g % NSTAGE], (g / NSTAGE) & 1);
        }
    }
    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(S.tmem_base, TMEM_COLS);
}

template <int NPASS>
__device__ __forceinline__ void compute_tq_all(const float *__restrict__ P, Smem<NPASS> &S, int ns) {
    compute_tq(P, S.times, ns, S.scratch, S.tq);
}

template <int NPASS>
__device__ __forceinline__ void begin_tile(Smem<NPASS> &S, State &st, const float *__restrict__ proj, int r0, int N, int rpo) {
    if (st.tile_r0 == r0) return;
    st.tile_r0 = r0;
    st.rpo = rpo;
    st.nrows = max(0, min(RT, N - r0));
    const int tid = threadIdx.x;
    const int first = r0 / rpo, last = (min(r0 + RT, N) - 1) / rpo;
    st.slot_base = first;
    st.nslots = r0 < N ? last - first + 1 : 0;
    if (st.nslots <= SLOTS) {
        const float4 *src = reinterpret_cast<const float4 *>(proj + (size_t)first * 768);
        float4 *dst = reinterpret_cast<float4 *>(S.pj);
        for (int i = tid; i < st.nslots * 192; i += NTHREADS) dst[i] = __ldg(src + i);
    }
}

// f_theta for the 128 rows in S.x -> S.x [r*9 + c]; `tq` is this stage's t-branch (768 floats in shared memory).
// All 320 threads call; ends with __syncthreads().
template <int NPASS>
__device__ __noinline__ void forward(const float *__restrict__ P, const float *__restrict__ proj, Smem<NPASS> &S,
                                     State &st, const float *tq) {
    constexpr int EPE = Smem<NPASS>::ENTRIES;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t tmem = S.tmem_base;
    const uint32_t eph = st.evals & 1;
    const int r0 = st.tile_r0;
    const long long t_begin = clock64();

    if (warp == 0) {
        // ---------------- TMA producer ----------------
        if (lane == 0) {
            for (int i = 0; i < EPE; ++i) {
                const uint32_t L = st.loads;
                mbar_wait(&S.empty[L % NSTAGE], ((L / NSTAGE) + 1) & 1);
                issue_entry<NPASS>(S, P, L);
                st.loads = L + 1;
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---------------- MMA issuer ----------------
        if (lane == 0) {
            const uint32_t a_hi = tmem + COL_A_HI, a_lo = tmem + COL_A_LO;
            // one weight chunk (hi image, then lo image in split mode) against k-atom `kc` of the A operand
            // (`nk` 16-wide k steps = 8 packed TMEM columns each) into accumulator columns d .. d + 127
            auto chunk = [&](uint32_t d, int kc, int nk, bool first) {
                if constexpr (NPASS == 2) {
                    // tf32: image w holds k 32 w .. 32 w + 31 of the k-atom; `nk` 16-wide k steps = 2 nk K = 8 MMAs
                    for (int w = 0; w < 2; ++w) {
                        const uint32_t g = st.consumed, s = g % NSTAGE;
                        mbar_wait(&S.full[s], (g / NSTAGE) & 1);
                        tc_fence_after();
                        const uint32_t b = smem_u32(&S.ring[s][0]);
                        for (int kk = 0; kk < 4 && 4 * w + kk < 2 * nk; ++kk)
                            umma_tf32_ts(d, a_hi + (uint32_t)(kc * 64 + w * 32 + kk * 8), make_desc(b + kk * 32), kIdescT128,
                                         (first && w == 0 && kk == 0) ? 0u : 1u);
                        umma_commit(&S.empty[s]);
                        st.consumed = g + 1;
                    }
                    return;
                }
                {
                    const uint32_t g = st.consumed, s = g % NSTAGE;
                    mbar_wait(&S.full[s], (g / NSTAGE) & 1);
                    tc_fence_after();
                    const uint32_t b = smem_u32(&S.ring[s][0]);
                    for (int kk = 0; kk < nk; ++kk) {
                        const uint32_t ac = (uint32_t)(kc * 32 + kk * 8);
                        umma_bf16_ts(d, a_hi + ac, make_desc(b + kk * 32), kIdescN128, (first && kk == 0) ? 0u : 1u);
                        if (NPASS == 3) umma_bf16_ts(d, a_lo + ac, make_desc(b + kk * 32), kIdescN128, 1u);
                    }
                    umma_commit(&S.empty[s]);
                    st.consumed = g + 1;
                }
                if (NPASS == 3) {
                    const uint32_t g = st.consumed, s = g % NSTAGE;
                    mbar_wait(&S.full[s], (g / NSTAGE) & 1);
                    tc_fence_after();
                    const uint32_t b = smem_u32(&S.ring[s][0]);
                    for (int kk = 0; kk < nk; ++kk)
                        umma_bf16_ts(d, a_hi + (uint32_t)(kc * 32 + kk * 8), make_desc(b + kk * 32), kIdescN128, 1u);
                    umma_commit(&S.empty[s]);
                    st.consumed = g + 1;
                }
            };
            const uint32_t acc = tmem + COL_ACC;
            // pose_encoder.0: K = 16 (9 used) -> D0 (both slots)
            mbar_wait(&S.a_ready, st.a_phase); st.a_phase ^= 1;
            tc_fence_after();
            chunk(acc, 0, 1, true);
            chunk(acc + 128, 0, 1, true);
            umma_commit(&S.dbar[0]);
            // pose_encoder.2 -> D1 (both slots; D0 has been read out by the time h1 is ready)
            mbar_wait(&S.a_ready, st.a_phase); st.a_phase ^= 1;
            tc_fence_after();
            for (int kc = 0; kc < 4; ++kc)
                for (int nh = 0; nh < 2; ++nh) chunk(acc + nh * 128, kc, 4, kc == 0);
            umma_commit(&S.dbar[1]);
            // heads: six half-heads alternate between the two accumulator slots
            mbar_wait(&S.a_ready, st.a_phase); st.a_phase ^= 1;
            tc_fence_after();
            for (int i = 0; i < 6; ++i) {
                if (i >= 2) { mbar_wait(&S.drain[i - 2], eph); tc_fence_after(); }   // the slot's previous half-head has been read out
                const uint32_t d = acc + (i & 1) * 128;
                for (int kc = 0; kc < 4; ++kc) chunk(d, kc, 4, kc == 0);
                umma_commit(&S.hbar[i]);
            }
        }
        __syncwarp();
    } else {
        // ---------------- epilogue warps ----------------
        const int e = warp - 2;
        const int row = 32 * (warp & 3) + lane;   // TMEM lane quarter is fixed by warp % 4
        const int half = e >> 2;                  // column half 0 / 1
        const uint32_t lane_addr = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
        extern __shared__ __align__(16) unsigned char gp_dyn_smem[];
        const uint32_t dyn0 = smem_u32(gp_dyn_smem);
        const float *sx = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.x) - dyn0));
        const float *sb1 = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.b1) - dyn0));
        const float *sb2 = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.b2) - dyn0));
        const float *spj = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.pj) - dyn0));
        const float *stq = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(tq) - dyn0));
        const float4 *swo = reinterpret_cast<const float4 *>(gp_dyn_smem + (smem_u32(S.wo) - dyn0));
        float *sxw = reinterpret_cast<float *>(gp_dyn_smem + (smem_u32(S.x) - dyn0));
        float *scratch = reinterpret_cast<float *>(gp_dyn_smem + (smem_u32(S.scratch) - dyn0));

        long long t0 = clock64();
        // inputs -> A operand: k 0..8 (k 9..15 zero), one row per thread of the first four epilogue warps
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

        // h1 = relu(D0 + b1) -> A
        mbar_wait(&S.dbar[0], eph);
        tc_fence_after();
        epi_hidden_t<NPASS>(lane_addr, COL_ACC, sb1, half * 128);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.a_ready);
        { const long long t1 = clock64(); st.cyc_l1 += t1 - t0; t0 = t1; }
        // h2 = relu(D1 + b2) -> A
        mbar_wait(&S.dbar[1], eph);
        tc_fence_after();
        { const long long t1 = clock64(); st.cyc_wait1 += t1 - t0; t0 = t1; }
        epi_hidden_t<NPASS>(lane_addr, COL_ACC, sb2, half * 128);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&S.a_ready);
        { const long long t1 = clock64(); st.cyc_epi1 += t1 - t0; t0 = t1; }

        // heads: z = relu(H + proj + tq), out = z . Wo^T over this thread's 64 columns of each half-head
        const int o = row < st.nrows ? (r0 + row) / st.rpo : -1;
        const bool use_pj = st.nslots <= SLOTS;
        const float *pjrow = spj + (use_pj && o >= 0 ? o - st.slot_base : 0) * 768;
        const float *prow = proj + (size_t)(o < 0 ? 0 : o) * 768;
        float acc[9];
#pragma unroll
        for (int c = 0; c < 9; ++c) acc[c] = 0.f;
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const int h = i >> 1, nh = i & 1;
            mbar_wait(&S.hbar[i], eph);
            tc_fence_after();
            { const long long t1 = clock64(); st.cyc_waith += t1 - t0; t0 = t1; }
            const int cb = h * 256 + nh * 128 + half * 64;   // first head column (0..767) of this thread
            const uint32_t taddr = lane_addr + COL_ACC + (i & 1) * 128 + half * 64;
            float a0 = 0.f, a1 = 0.f, a2 = 0.f;
            uint32_t r[2][32];
            tmem_ld32_nowait(taddr, r[0]);
            tmem_ld32_nowait(taddr + 32, r[1]);
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                tmem_ld_wait();
#pragma unroll
                for (int j8 = 0; j8 < 4; ++j8) {
                    const int c0 = cb + g * 32 + j8 * 8;
                    float4 w[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) w[j] = swo[c0 + j];
                    const float4 ta = *reinterpret_cast<const float4 *>(stq + c0);
                    const float4 tb = *reinterpret_cast<const float4 *>(stq + c0 + 4);
                    const float *ebase = use_pj ? pjrow + c0 : prow + c0;
                    const float4 ea = *reinterpret_cast<const float4 *>(ebase);
                    const float4 eb = *reinterpret_cast<const float4 *>(ebase + 4);
                    const float ev[8] = {ea.x + ta.x, ea.y + ta.y, ea.z + ta.z, ea.w + ta.w,
                                         eb.x + tb.x, eb.y + tb.y, eb.z + tb.z, eb.w + tb.w};
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        const float z = fmaxf(__uint_as_float(r[g][j8 * 8 + j]) + ev[j], 0.f);
                        a0 = fmaf(z, w[j].x, a0); a1 = fmaf(z, w[j].y, a1); a2 = fmaf(z, w[j].z, a2);
                    }
                }
            }
            acc[h * 3 + 0] += a0; acc[h * 3 + 1] += a1; acc[h * 3 + 2] += a2;
            if (i < 4) {   // this slot has been read out: the MMA warp may overwrite it with half-head i + 2
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(&S.drain[i]);
            }
            { const long long t1 = clock64(); st.cyc_epi2 += t1 - t0; t0 = t1; }
        }
        tc_fence_before();
        // the two column halves of a row meet through shared memory; half 0 writes the output tile
        if (half == 1) {
#pragma unroll
            for (int c = 0; c < 9; ++c) scratch[c * RT + row] = acc[c];
        }
        asm volatile("bar.sync 1, 256;" ::: "memory");  // the 8 epilogue warps only
        if (half == 0) {
            const float *sbo = reinterpret_cast<const float *>(gp_dyn_smem + (smem_u32(S.bo) - dyn0));
#pragma unroll
            for (int c = 0; c < 9; ++c) sxw[row * XS + c] = (acc[c] + scratch[c * RT + row]) + sbo[c];
        }
        st.cyc_tail += clock64() - t0;
    }
    __syncthreads();
    st.evals += 1;
    st.cyc_fwd += clock64() - t_begin;
}

}  // namespace solot
}  // namespace gp
