// Layers 2 and 3 of a PointNet++ set-abstraction scale and its max-pool in ONE persistent tensor-core kernel
// (P2/pointnet2_modules.py:45-66 on the rows produced by P2/pointnet2_utils.py:279-296):
//
//   A[r][k] = relu(P[batch(r) * n_src + gidx[r]][k] - Q[r / q_ns][k])          hoisted first layer, applied on the fly
//   H       = relu(A . W1^T + b1)                                              [128 rows x c2], never leaves the SM
//   out[g]  = max over the pool_ns rows of group g of relu(H . W2^T + b2)      [rows / pool_ns, c3]
//
// The (centre, sample) activation matrices of the reference -- c2 and c3 floats for each of B*npoint*nsample
// rows -- never exist in HBM.  Per 128-row tile:
//   gather   worker warps read P rows by ball-query index (coalesced: 16 lanes per row), subtract Q, ReLU, split to
//            bf16 (hi / lo) and store swizzled A-operand atoms in shared memory;
//   GEMM 1   A (shared memory) x W1 chunks -> D (TMEM);
//   hidden   H = relu(D + b1) -> packed bf16 pairs written straight into TENSOR MEMORY (tcgen05.st): the second GEMM
//            takes its A operand from TMEM (tcgen05.mma [d], [a_tmem], b_desc), so H never touches shared memory;
//   GEMM 2   H (TMEM) x W2 chunks -> D (TMEM, the same columns: D of GEMM 1 has been read out);
//   pool     max over the pool_ns rows of each group = over lanes of a warp (row = TMEM lane): a recursive-halving
//            butterfly in registers (31 shuffles per 32 x 32 block), bias + ReLU once per pooled value
//            (relu(max(x) + b) == max(relu(x + b)) bit for bit), coalesced stores.  No shared-memory staging.
// What the TMEM-resident H buys (round 2): the shared-memory A buffer only holds the GATHERED operand, which GEMM 1 has
// finished reading long before the tile is done -- so the worker warps gather tile t + 1 while the tensor pipe runs
// GEMM 2 of tile t (they used to idle there), the buffer is half as large at levels 3-4, and the freed shared memory
// deepens the weight ring (5-10 single 16 KB images instead of 2 hi+lo stages: the weight stream, ~1.3 k cycles round
// trip per image, was what bounded GEMM 2 at level 4).  Accumulators are processed in passes of at most 256 columns =
// two 128-column chunks whose MMA chains are issued interleaved (a chain into one accumulator retires one MMA per ~90
// cycles, an N = 128 MMA occupies the pipe for 64: two chains keep it busy).
//
// TMEM map: [0, hcols) H (hi: 32 columns per 64-wide k-atom, then lo in split mode; tf32: one column per k, 64 per
// k-atom) | [hcols, hcols + DN) accumulators.
// CTA = NW worker warps + producer + MMA issuer, persistent over tiles: warp 0 streams the weight chunks
// (cp.async.bulk, [<=128 n][64 k] images from the gp_gemm_pack layout) through a shared-memory ring and runs ahead
// across tiles; warp 1 issues the MMAs; warps 2.. gather / convert / run both epilogues.
// NPASS = 1: bf16 operands; NPASS = 3: split-bf16 (hi*hi + lo*hi + hi*lo), fp32-class; NPASS = 2: tf32 operands
// (rounded to nearest, tf32_rna_bits), kind::tf32 K = 8.  A tf32 64-k atom is two [rows][32 k] fp32 images (k 0..31, k 32..63) in the places of
// the hi and lo images, so the ring, A buffer and TMEM plans are those of the split mode; an image whose k range is
// beyond the layer's K (the second image of a K <= 32 layer) is neither streamed nor multiplied.
#include "common.cuh"
#include "tc_ptx.cuh"

#ifndef GP_SAF_ROW_MODE
#define GP_SAF_ROW_MODE 1
#endif

namespace gp {
namespace saf {

using namespace gp::tc;

constexpr int BM = 128;
constexpr int ATOM = 128 * 128;   // [128 rows][64 k] bf16
constexpr int SLOT = 128 * 128;   // ring slot: one weight image of up to [128 n][64 k] bf16
constexpr int MAX_NST = 12;

struct Args {
    const float *P;
    int n_src, ldp;
    const int *gidx;
    long long R;
    int rows_per_batch;
    const float *Q;
    int ldq, q_ns;
    const uint8_t *W1p;
    const float *b1;
    int c1, c2;
    const uint8_t *W2p;
    const float *b2;
    int c3;
    int pool_ns;
    float *pooled;
    int ld_pooled;
    int ntiles;
    // first-level mode (xyz != nullptr; P / Q unused): A[r][k] = relu(W0[k] . (xyz[batch(r)][gidx[r]] - centres[r / q_ns]) + b0[k]),
    // the K = 3 first layer evaluated in the operand loader
    const float *xyz;        // [batches, n_src, 3]
    const float *centres;    // [R / q_ns, 3]
    float w0c[64 * 3], b0c[64];   // folded first layer [c1][3], [c1]: travels in the launch's parameter space (constant operands)
    // launch configuration (host)
    int nst;             // ring slots
    int tmem_cols;       // allocated TMEM columns (256 or 512)
    int hcols;           // TMEM columns of H (hi + lo)
    int dn;              // accumulator columns per pass (128 or 256)
    int bias_smem;       // biases staged in shared memory (else read through L1)
    int tile_in_batch;   // rows_per_batch % 128 == 0: all rows of a tile belong to one batch
    int q_shift;         // log2(q_ns) if q_ns is a power of two, else -1
};

template <int NPASS>
struct Cfg {
    static constexpr int IMAGES = NPASS == 1 ? 1 : 2;
};
// whether image w of k-atom c of a layer with K = kdim takes part (the split mode's lo images always do)
template <int NPASS>
__host__ __device__ inline bool image_used(int kdim, int c, int w) { return NPASS != 2 || 64 * c + 32 * w < kdim; }

__host__ __device__ inline int round16(int n) { return (n + 15) & ~15; }
__host__ __device__ inline int atoms_of(int k) { return (k + 63) / 64; }

// shared memory carve-up (bytes from a 1024-aligned base): weight ring | gathered A buffer | biases | barriers
template <int NPASS>
struct Layout {
    int k1, nst, bias_smem;
    __host__ __device__ Layout(int c1, int nst_, int bias_smem_) : k1(atoms_of(c1)), nst(nst_), bias_smem(bias_smem_) {}
    __host__ __device__ size_t ring() const { return 0; }
    __host__ __device__ size_t abuf() const { return (size_t)nst * SLOT; }
    __host__ __device__ size_t abuf_bytes() const { return (size_t)Cfg<NPASS>::IMAGES * k1 * ATOM; }
    __host__ __device__ size_t bias() const { return abuf() + abuf_bytes(); }
    __host__ __device__ size_t bars() const { return bias() + (bias_smem ? (384 + 512) * sizeof(float) : 0); }
    __host__ __device__ size_t total() const { return bars() + 512 + 1024; }
};

// Max-pool of one warp's 32 rows (lane = row; -inf for rows that do not exist) x 32 columns of raw accumulators over
// groups of NS consecutive rows (= lanes), then bias + ReLU once per pooled value.  Recursive halving over the lanes of
// a group: at every butterfly step a lane keeps one half of its columns and hands the other half to its partner, so
// the 32 x 32 block is reduced with 31 shuffles per lane (not 32 x log2 NS) and without shared memory; lane l of a
// group ends up with the 32 / NS consecutive columns (l % NS) * 32 / NS .. of its group's pooled row (coalesced stores).
template <int NS>
__device__ __forceinline__ void pool_block(const uint32_t (&r)[32], bool row_ok, int lane, long long grow0, long long R,
                                           int nbase, int N, const float *bias, float *pooled, int ld_pooled, bool vec_ok) {
    float v[32];
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = row_ok ? __uint_as_float(r[j]) : -INFINITY;
#pragma unroll
    for (int bit = NS / 2, h = 16; bit >= 1; bit >>= 1, h >>= 1) {
        const bool up = (lane & bit) != 0;
#pragma unroll
        for (int j = 0; j < h; ++j) {
            const float mine = up ? v[j + h] : v[j];
            const float theirs = up ? v[j] : v[j + h];
            v[j] = fmaxf(mine, __shfl_xor_sync(0xffffffffu, theirs, bit));
        }
    }
    constexpr int KEEP = 32 / NS;                 // consecutive columns this lane ends up with
    const int grp = lane / NS;                    // pooled row of this lane's group inside the 32-row block
    const long long prow = grow0 / NS + grp;
    if (grow0 + (long long)grp * NS < R) {
        const int n0 = nbase + (lane & (NS - 1)) * KEEP;
        float *dst = pooled + prow * (long long)ld_pooled + n0;
        float o[KEEP];
#pragma unroll
        for (int i = 0; i < KEEP; ++i) o[i] = n0 + i < N ? fmaxf(v[i] + bias[n0 + i], 0.f) : 0.f;
        // a lane's KEEP columns are consecutive: one 8- / 16-byte store when the row allows it
        if (KEEP == 2 && vec_ok && n0 + 1 < N) {
            *reinterpret_cast<float2 *>(dst) = make_float2(o[0], o[1]);
        } else if (KEEP == 4 && vec_ok && n0 + 3 < N) {
            *reinterpret_cast<float4 *>(dst) = make_float4(o[0], o[1], o[2], o[3]);
        } else {
#pragma unroll
            for (int i = 0; i < KEEP; ++i)
                if (n0 + i < N) dst[i] = o[i];
        }
    }
}

// First-level mode: one thread = one row.  x[k] = relu(W0[k] . d + b0[k]) for the thread's C1 / PARTS output channels
// (weights from the parameter space: uniform operands), split to bf16 hi / lo (or rounded to tf32) and stored as
// 16-byte chunks of the swizzled A operand atom.
template <int NPASS, int C1, int PARTS>
__device__ __forceinline__ void xyz_first_layer(const Args &a, int part, float dx, float dy, float dz, bool valid, int rl,
                                                uint32_t A_hi, uint32_t A_lo) {
    constexpr int NC = C1 / PARTS;
    static_assert(NC % 8 == 0, "a thread writes whole 16-byte chunks");
#pragma unroll
    for (int c8 = 0; c8 < NC / 8; ++c8) {
        float x[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int k = part * NC + c8 * 8 + j;
            // same operation order as the FP32 level-1 kernel (dense_relu_c): ((b + dx w0) + dy w1) + dz w2
            const float v = fmaf(dz, a.w0c[k * 3 + 2], fmaf(dy, a.w0c[k * 3 + 1], fmaf(dx, a.w0c[k * 3], a.b0c[k])));
            x[j] = valid ? fmaxf(v, 0.f) : 0.f;
        }
        if (NPASS == 2) {   // C1 <= 32: image 0 only, 4 k per 16 bytes
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j16 = (part * NC + c8 * 8) / 4 + h;
                const uint32_t off = rl * 128 + ((j16 ^ (rl & 7)) << 4);
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(A_hi + off), "r"(tf32_rna_bits((x[4 * h]))),
                             "r"(tf32_rna_bits((x[4 * h + 1]))), "r"(tf32_rna_bits((x[4 * h + 2]))),
                             "r"(tf32_rna_bits((x[4 * h + 3]))));
            }
            continue;
        }
        const int j16 = (part * NC) / 8 + c8;
        const uint32_t off = rl * 128 + ((j16 ^ (rl & 7)) << 4);
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const __nv_bfloat162 h = __floats2bfloat162_rn(x[2 * j], x[2 * j + 1]);
            hi[j] = *reinterpret_cast<const uint32_t *>(&h);
            if (NPASS == 3) {
                const float2 f = __bfloat1622float2(h);
                const __nv_bfloat162 l = __floats2bfloat162_rn(x[2 * j] - f.x, x[2 * j + 1] - f.y);
                lo[j] = *reinterpret_cast<const uint32_t *>(&l);
            }
        }
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(A_hi + off), "r"(hi[0]), "r"(hi[1]), "r"(hi[2]), "r"(hi[3]));
        if (NPASS == 3)
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(A_lo + off), "r"(lo[0]), "r"(lo[1]), "r"(lo[2]), "r"(lo[3]));
    }
}

// NW worker warps (gather / convert / epilogues) + producer + MMA issuer.  NW = 8: one CTA per SM; NW = 4: 192-thread
// CTAs, two per SM when a CTA needs at most half of the shared memory and 256 TMEM columns.
template <int NPASS, int NW>
__global__ void __launch_bounds__((NW + 2) * 32, NW == 4 ? 2 : 1) sa_mlp2_kernel(const __grid_constant__ Args a) {
    using C = Cfg<NPASS>;
    constexpr int IM = C::IMAGES;
    constexpr int NTHREADS = (NW + 2) * 32;
    constexpr int HALVES = NW / 4;          // worker warps per TMEM lane quarter: they split the 32-column groups
    constexpr int RSTEP = 2 * NW;           // rows covered by one gather pass (16 lanes per row)
    constexpr int RP = 128 / RSTEP;         // rows of a tile per worker thread
    const int NST = a.nst;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint8_t *base = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const Layout<NPASS> L(a.c1, a.nst, a.bias_smem);
    uint8_t *ring = base + L.ring();
    uint8_t *abuf = base + L.abuf();
    float *sb1 = reinterpret_cast<float *>(base + L.bias());
    float *sb2 = sb1 + 384;
    const float *b1p = a.bias_smem ? sb1 : a.b1, *b2p = a.bias_smem ? sb2 : a.b2;   // valid for n < c2 / n < c3
    unsigned long long *bars = reinterpret_cast<unsigned long long *>(base + L.bars());
    unsigned long long *full = bars, *empty = bars + MAX_NST;
    unsigned long long *a_ready = bars + 2 * MAX_NST;       // gathered rows of the next tile are in the A buffer (NW arrivals)
    unsigned long long *d1bar = a_ready + 1;                // a pass of GEMM 1 is complete (commit)
    unsigned long long *e1_done = a_ready + 2;              // that pass has been read out into H (NW arrivals)
    unsigned long long *d2bar = a_ready + 3;                // a pass of GEMM 2 is complete (commit)
    unsigned long long *p_done = a_ready + 4;               // that pass has been pooled (NW arrivals)
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(a_ready + 5);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int k1 = atoms_of(a.c1), k2 = atoms_of(a.c2);
    const int bn1 = round16(a.c2), bn2 = round16(a.c3);
    const int DN = a.dn;
    const int np1 = (bn1 + DN - 1) / DN, np2 = (bn2 + DN - 1) / DN;     // accumulator passes of the two GEMMs
    const int my_tiles = a.ntiles > (int)blockIdx.x ? (a.ntiles - 1 - (int)blockIdx.x) / (int)gridDim.x + 1 : 0;

    if (tid == 0) {
        for (int s = 0; s < NST; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        mbar_init(a_ready, NW);
        mbar_init(d1bar, 1);
        mbar_init(e1_done, NW);
        mbar_init(d2bar, 1);
        mbar_init(p_done, NW);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (a.bias_smem) {
        for (int i = tid; i < 512; i += NTHREADS) {
            if (i < 384) sb1[i] = i < a.c2 ? __ldg(a.b1 + i) : 0.f;
            sb2[i] = i < a.c3 ? __ldg(a.b2 + i) : 0.f;
        }
    }
    __syncthreads();
    if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)a.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = *tmem_slot;
    const uint32_t abuf_a = smem_u32(abuf);
    const uint32_t h_hi = tmem, h_lo = tmem + (uint32_t)(k2 * 32);   // H: 32 packed columns per k-atom
    const uint32_t dcol = (uint32_t)a.hcols;                         // accumulators start after H

    // number of 128-column chunks of pass `p` of a GEMM whose (rounded) width is bn, and the rows (= columns) of chunk nh
    auto pass_chunks = [&](int bn, int p) { const int w = min(DN, bn - p * DN); return (w + 127) / 128; };
    auto chunk_rows = [&](int bn, int p, int nh) { return min(128, bn - p * DN - nh * 128); };

    if (warp == 0) {
        // ---------------- weight producer ----------------
        // entry order per tile = consumption order: GEMM 1 passes, then GEMM 2 passes; per pass: k-atom c, image
        // (hi, lo), chunk nh
        if (lane == 0) {
            uint32_t slot = 0, wrap = 0;   // ring position of the next entry; `wrap` = how often the ring has been filled
#ifdef GP_SAF_PROBE
            long long pw = 0, pt0 = clock64(), nent = 0;
#endif
            for (int t = 0; t < my_tiles; ++t) {
                for (int gm = 0; gm < 2; ++gm) {
                    const uint8_t *wp = gm ? a.W2p : a.W1p;
                    const int bn = gm ? bn2 : bn1, kat = gm ? k2 : k1, np = gm ? np2 : np1;
                    for (int p = 0; p < np; ++p) {
                        const int nch = pass_chunks(bn, p);
                        for (int c = 0; c < kat; ++c)
                            for (int w = 0; w < IM; ++w) {
                                if (!image_used<NPASS>(gm ? a.c2 : a.c1, c, w)) continue;
                                for (int nh = 0; nh < nch; ++nh) {
#ifdef GP_SAF_PROBE
                                    const long long w0 = clock64();
                                    ++nent;
#endif
                                    if (wrap) mbar_wait(&empty[slot], (wrap + 1) & 1);
#ifdef GP_SAF_PROBE
                                    pw += clock64() - w0;
#endif
                                    // gp_gemm_pack layout: n-tiles of 256 columns, per tile and k-chunk one image
                                    // [bn_tile x 128 B] (hi, lo)
                                    const int ncol = p * DN + nh * 128, jt = ncol >> 8, within = ncol & 255;
                                    const int bnj = min(256, bn - 256 * jt);
                                    const uint32_t rows = (uint32_t)chunk_rows(bn, p, nh);
                                    const size_t img = (size_t)bnj * 128;
                                    const uint8_t *tile = wp + (size_t)jt * kat * IM * (256 * 128);
                                    mbar_arrive_expect_tx(&full[slot], rows * 128);
                                    bulk_g2s(ring + (size_t)slot * SLOT, tile + ((size_t)c * IM + w) * img + (size_t)within * 128,
                                             rows * 128, &full[slot]);
                                    if (++slot == (uint32_t)NST) { slot = 0; ++wrap; }
                                }
                            }
                    }
                }
            }
#ifdef GP_SAF_PROBE
            if (blockIdx.x == 0 && my_tiles)
                printf("saf producer: entries/tile %lld, cycles/tile %lld of which waiting for a free slot %lld (nst %d)\n", nent / my_tiles,
                       (clock64() - pt0) / my_tiles, pw / my_tiles, NST);
#endif
        }
        __syncwarp();
    } else if (warp == 1) {
        // ---------------- MMA issuer ----------------
        // The whole warp runs this code with identical state; one elected lane issues each MMA / commit (tc_ptx.cuh).
        {
            const uint32_t a_hi = abuf_a, a_lo = abuf_a + (NPASS != 1 ? k1 * ATOM : 0);
            const uint32_t ring_a = smem_u32(ring);
            uint32_t slot = 0, fph = 0;     // ring position of the next entry to consume, parity of its `full` barrier
            uint32_t ph_a = 0, ph_e1 = 0, ph_p = 0;
#ifdef GP_SAF_PROBE
            long long mw_full = 0, mw_other = 0, mt0 = clock64();
#endif
            // Everything the MMA thread touches stays in (uniform) registers: no arrays, no 64-bit arithmetic -- an MMA
            // whose descriptors come from local memory is issued through a R2UR waterfall, ~400 cycles apiece.
            // next ring entry: wait for it, return its shared-memory address; `done` hands it back to the producer
            auto take = [&](uint32_t &s_out) -> uint32_t {
                const uint32_t sl = slot;
                mbar_wait(&full[sl], fph);
                if (++slot == (uint32_t)NST) { slot = 0; fph ^= 1; }
                s_out = sl;
                return ring_a + sl * SLOT;
            };
            // one accumulator pass: kat k-atoms, one or two chunks of <= 128 columns (two chunks = two interleaved chains)
            // `kdim`: the populated K (c1 / c2): the last k-atom multiplies only its populated 16-wide (tf32: 8-wide) steps
            auto pass = [&](const bool second, const int kat, const int kdim, const int bn, const int p) {
                const bool two = pass_chunks(bn, p) == 2;
                const uint32_t id0 = NPASS == 2 ? make_idesc_tf32(128, (uint32_t)chunk_rows(bn, p, 0))
                                                : make_idesc_bf16(128, (uint32_t)chunk_rows(bn, p, 0));
                const uint32_t id1 = two ? (NPASS == 2 ? make_idesc_tf32(128, (uint32_t)chunk_rows(bn, p, 1))
                                                       : make_idesc_bf16(128, (uint32_t)chunk_rows(bn, p, 1))) : id0;
                const uint32_t d0 = tmem + dcol, d1 = d0 + 128;
                if (NPASS == 2) {
                    // image w of atom c: k 64 c + 32 w .. +31; A from the A buffer's image or from H's columns k
                    for (int c = 0; c < kat; ++c)
                        for (int w = 0; w < 2; ++w) {
                            if (!image_used<NPASS>(kdim, c, w)) break;
                            uint32_t s0 = 0, s1 = 0, b0, b1 = 0;
                            b0 = take(s0);
                            if (two) b1 = take(s1);
                            tc_fence_after();
                            const int k0 = 64 * c + 32 * w;
                            const int nk = min(4, (kdim - k0 + 7) >> 3);
                            for (int kk = 0; kk < nk; ++kk) {
                                const uint32_t accum = (c | w | kk) ? 1u : 0u;
                                if (second) {
                                    const uint32_t ah = h_hi + k0 + kk * 8;
                                    umma_tf32_ts_w(d0, ah, make_desc(b0 + kk * 32), id0, accum);
                                    if (two) umma_tf32_ts_w(d1, ah, make_desc(b1 + kk * 32), id1, accum);
                                } else {
                                    const uint64_t ad = make_desc((w ? a_lo : a_hi) + c * ATOM + kk * 32);
                                    umma_tf32_ss_w(d0, ad, make_desc(b0 + kk * 32), id0, accum);
                                    if (two) umma_tf32_ss_w(d1, ad, make_desc(b1 + kk * 32), id1, accum);
                                }
                            }
                            umma_commit_w(&empty[s0]);
                            if (two) umma_commit_w(&empty[s1]);
                        }
                    return;
                }
                for (int c = 0; c < kat; ++c) {
                    uint32_t s0 = 0, s1 = 0, b0, b1 = 0;
#ifdef GP_SAF_PROBE
                    long long w0 = clock64();
#endif
                    b0 = take(s0);            // hi images of the chunk(s)
                    if (two) b1 = take(s1);
                    tc_fence_after();
#ifdef GP_SAF_PROBE
                    mw_full += clock64() - w0;
#endif
                    const int nk = min(4, (kdim - 64 * c + 15) >> 4);
                    for (int kk = 0; kk < nk; ++kk) {
                        const uint32_t accum = (c | kk) ? 1u : 0u;
                        const uint32_t ah = second ? h_hi + c * 32 + kk * 8 : a_hi + c * ATOM + kk * 32;
                        const uint32_t al = second ? h_lo + c * 32 + kk * 8 : a_lo + c * ATOM + kk * 32;
                        if (second) {
                            umma_bf16_ts_w(d0, ah, make_desc(b0 + kk * 32), id0, accum);
                            if (two) umma_bf16_ts_w(d1, ah, make_desc(b1 + kk * 32), id1, accum);
                            if (NPASS == 3) {
                                umma_bf16_ts_w(d0, al, make_desc(b0 + kk * 32), id0, 1u);
                                if (two) umma_bf16_ts_w(d1, al, make_desc(b1 + kk * 32), id1, 1u);
                            }
                        } else {
                            umma_bf16_w(d0, make_desc(ah), make_desc(b0 + kk * 32), id0, accum);
                            if (two) umma_bf16_w(d1, make_desc(ah), make_desc(b1 + kk * 32), id1, accum);
                            if (NPASS == 3) {
                                umma_bf16_w(d0, make_desc(al), make_desc(b0 + kk * 32), id0, 1u);
                                if (two) umma_bf16_w(d1, make_desc(al), make_desc(b1 + kk * 32), id1, 1u);
                            }
                        }
                    }
                    umma_commit_w(&empty[s0]);
                    if (two) umma_commit_w(&empty[s1]);
                    if (NPASS == 3) {
#ifdef GP_SAF_PROBE
                        w0 = clock64();
#endif
                        b0 = take(s0);        // lo images
                        if (two) b1 = take(s1);
                        tc_fence_after();
#ifdef GP_SAF_PROBE
                        mw_full += clock64() - w0;
#endif
                        for (int kk = 0; kk < nk; ++kk) {
                            const uint32_t ah = second ? h_hi + c * 32 + kk * 8 : a_hi + c * ATOM + kk * 32;
                            if (second) {
                                umma_bf16_ts_w(d0, ah, make_desc(b0 + kk * 32), id0, 1u);
                                if (two) umma_bf16_ts_w(d1, ah, make_desc(b1 + kk * 32), id1, 1u);
                            } else {
                                umma_bf16_w(d0, make_desc(ah), make_desc(b0 + kk * 32), id0, 1u);
                                if (two) umma_bf16_w(d1, make_desc(ah), make_desc(b1 + kk * 32), id1, 1u);
                            }
                        }
                        umma_commit_w(&empty[s0]);
                        if (two) umma_commit_w(&empty[s1]);
                    }
                }
            };
            for (int t = 0; t < my_tiles; ++t) {
#ifdef GP_SAF_PROBE
                const long long w0 = clock64();
#endif
                mbar_wait(a_ready, ph_a); ph_a ^= 1;        // gathered rows of tile t are in the A buffer
                tc_fence_after();
#ifdef GP_SAF_PROBE
                mw_other += clock64() - w0;
#endif
                for (int p = 0; p < np1; ++p) {
                    if (p > 0) { mbar_wait(e1_done, ph_e1); ph_e1 ^= 1; tc_fence_after(); }   // accumulators read out
                    pass(false, k1, a.c1, bn1, p);
                    umma_commit_w(d1bar);
                }
                mbar_wait(e1_done, ph_e1); ph_e1 ^= 1;     // H is complete in TMEM, accumulators free
                tc_fence_after();
                for (int q = 0; q < np2; ++q) {
                    if (q > 0) { mbar_wait(p_done, ph_p); ph_p ^= 1; tc_fence_after(); }
                    pass(true, k2, a.c2, bn2, q);
                    umma_commit_w(d2bar);
                }
                mbar_wait(p_done, ph_p); ph_p ^= 1;        // last pass pooled: accumulators free for the next tile
                tc_fence_after();
            }
#ifdef GP_SAF_PROBE
            if (blockIdx.x == 0 && my_tiles && lane == 0)
                printf("saf mma: cycles/tile %lld, waiting for weights %lld, waiting for a_ready %lld\n", (clock64() - mt0) / my_tiles,
                       mw_full / my_tiles, mw_other / my_tiles);
#endif
        }
        __syncwarp();
    } else {
        // ---------------- gather / convert / epilogues ----------------
        const int w = tid - 64;                    // 0..32 NW - 1
        const int e = warp - 2;
        const int quarter = warp & 3;              // TMEM lane quarter of this warp
        const int half = e >> 2;                   // which 32-column groups (odd / even)
        const int row = 32 * quarter + lane;       // epilogue row
        const uint32_t lane_addr = tmem + ((uint32_t)(32 * quarter) << 16);
        const uint32_t A_hi = abuf_a, A_lo = abuf_a + (NPASS != 1 ? k1 * ATOM : 0);
        const int jv = w & 15;                     // float4 inside a 64-float chunk
        const int rsub = w >> 4;                   // row inside a pass
        const int ns = a.pool_ns;
        // pooled rows can take 16-byte vector stores (every row start and every 32-column block is 16-byte aligned)
        const bool vec_ok = (reinterpret_cast<uintptr_t>(a.pooled) & 15) == 0 && (a.ld_pooled & 3) == 0;
        // Rows rsub + RSTEP p (p < RP) of a tile belong to this thread's gather.  Their ball-query indices for the
        // next tile are requested early and only consumed at the gather: the index load is the head of the gather's
        // latency chain.
        int gi[RP];
        int gx = -1;     // one-row-per-thread loaders: the ball-query index of THIS thread's row (row w % 128 of the tile)
        // a single k-atom (c1 <= 64): one thread converts one whole row (its 8 / HALVES 16-byte chunks) -- per-row address
        // arithmetic once instead of once per 16 lanes
        const bool row_mode = !a.xyz && k1 == 1 && GP_SAF_ROW_MODE;
        auto request = [&](int t) {
            const long long row0 = ((long long)blockIdx.x + (long long)t * gridDim.x) * BM;
            if (a.xyz || row_mode) {
                const long long gr = row0 + (w & 127);
                gx = -1;
                if (t < my_tiles && gr < a.R) asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(gx) : "l"(a.gidx + gr));
                return;
            }
#pragma unroll
            for (int p = 0; p < RP; ++p) {
                const long long gr = row0 + rsub + RSTEP * p;
                gi[p] = -1;
                if (t < my_tiles && gr < a.R) asm volatile("ld.global.nc.s32 %0, [%1];" : "=r"(gi[p]) : "l"(a.gidx + gr));
            }
        };
        // gather k-atoms [kc_lo, kc_hi) of tile t into the A buffer (its indices are in gi[]): thread handles rows
        // rsub + RSTEP p (p < RP), 16 bytes of every 64-float chunk, 8 rows at a time; `last` publishes the tile
        // first-level mode: one row per thread (all NW * 32 worker threads: with 8 worker warps two threads split a row's channels)
        auto gather_xyz = [&](int t) {
            const long long row0 = ((long long)blockIdx.x + (long long)t * gridDim.x) * BM;
            const int rl = w & 127, part = w >> 7;
            const int g32 = (int)(row0 + rl);
            const bool valid = gx >= 0;
            float dx = 0.f, dy = 0.f, dz = 0.f;
            if (valid) {
                const int batch = g32 / a.rows_per_batch;
                const int qrow = a.q_shift >= 0 ? g32 >> a.q_shift : g32 / a.q_ns;
                const float *pt = a.xyz + ((long long)batch * a.n_src + gx) * 3;
                const float *ct = a.centres + (long long)qrow * 3;
                dx = __ldg(pt) - __ldg(ct); dy = __ldg(pt + 1) - __ldg(ct + 1); dz = __ldg(pt + 2) - __ldg(ct + 2);
            }
            if (a.c1 == 32) xyz_first_layer<NPASS, 32, HALVES>(a, part, dx, dy, dz, valid, rl, A_hi, A_lo);
            else xyz_first_layer<NPASS, 16, HALVES>(a, part, dx, dy, dz, valid, rl, A_hi, A_lo);
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(a_ready);
        };
        auto gather_row = [&](int t) {
            const long long row0 = ((long long)blockIdx.x + (long long)t * gridDim.x) * BM;
            const int rl = w & 127, part = w >> 7;
            const int g32 = (int)(row0 + rl);
            constexpr int NCH = 8 / HALVES;          // 16-byte bf16 chunks (8 columns) of this thread
            float4 pv[NCH][2], qv[NCH][2];
            const bool valid = gx >= 0;
            const int batch = g32 / a.rows_per_batch;
            const int qrow = a.q_shift >= 0 ? g32 >> a.q_shift : g32 / a.q_ns;
            const float *prow = a.P + ((long long)batch * a.n_src + (valid ? gx : 0)) * a.ldp + part * NCH * 8;
            const float *qrowp = a.Q + (long long)(valid ? qrow : 0) * a.ldq + part * NCH * 8;
#pragma unroll
            for (int c = 0; c < NCH; ++c)
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const bool ok = valid && part * NCH * 8 + c * 8 + h * 4 < a.c1;
                    pv[c][h] = ok ? __ldg(reinterpret_cast<const float4 *>(prow + c * 8 + h * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    qv[c][h] = ok ? __ldg(reinterpret_cast<const float4 *>(qrowp + c * 8 + h * 4)) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
            for (int c = 0; c < NCH; ++c) {
                const float x[8] = {fmaxf(pv[c][0].x - qv[c][0].x, 0.f), fmaxf(pv[c][0].y - qv[c][0].y, 0.f),
                                    fmaxf(pv[c][0].z - qv[c][0].z, 0.f), fmaxf(pv[c][0].w - qv[c][0].w, 0.f),
                                    fmaxf(pv[c][1].x - qv[c][1].x, 0.f), fmaxf(pv[c][1].y - qv[c][1].y, 0.f),
                                    fmaxf(pv[c][1].z - qv[c][1].z, 0.f), fmaxf(pv[c][1].w - qv[c][1].w, 0.f)};
                if (NPASS == 2) {   // column col = part NCH 8 + 8 c + 4 h: image col / 32, 16-byte unit (col % 32) / 4
#pragma unroll
                    for (int h = 0; h < 2; ++h) {
                        const int col = (part * NCH + c) * 8 + 4 * h;
                        const uint32_t off = (col >> 5) * (k1 * ATOM) + rl * 128 + ((((col & 31) >> 2) ^ (rl & 7)) << 4);
                        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(A_hi + off), "r"(tf32_rna_bits((x[4 * h]))),
                                     "r"(tf32_rna_bits((x[4 * h + 1]))), "r"(tf32_rna_bits((x[4 * h + 2]))),
                                     "r"(tf32_rna_bits((x[4 * h + 3]))));
                    }
                    continue;
                }
                const int j16 = part * NCH + c;
                const uint32_t off = rl * 128 + ((j16 ^ (rl & 7)) << 4);
                uint32_t hi[4], lo[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const __nv_bfloat162 h = __floats2bfloat162_rn(x[2 * j], x[2 * j + 1]);
                    hi[j] = *reinterpret_cast<const uint32_t *>(&h);
                    if (NPASS == 3) {
                        const float2 f = __bfloat1622float2(h);
                        const __nv_bfloat162 l = __floats2bfloat162_rn(x[2 * j] - f.x, x[2 * j + 1] - f.y);
                        lo[j] = *reinterpret_cast<const uint32_t *>(&l);
                    }
                }
                asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(A_hi + off), "r"(hi[0]), "r"(hi[1]), "r"(hi[2]), "r"(hi[3]));
                if (NPASS == 3)
                    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(A_lo + off), "r"(lo[0]), "r"(lo[1]), "r"(lo[2]), "r"(lo[3]));
            }
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) mbar_arrive(a_ready);
        };
        auto gather = [&](int t, int kc_lo, int kc_hi, bool last) {
            if (a.xyz || row_mode) {   // c1 <= 64: one k-atom, one part
                if (last) { if (a.xyz) gather_xyz(t); else gather_row(t); }
                return;
            }
            const long long row0 = ((long long)blockIdx.x + (long long)t * gridDim.x) * BM;
            const int tile_batch = (int)(row0 / a.rows_per_batch);
#pragma unroll
            for (int pb = 0; pb < RP; pb += 8) {
                long long src[8];
                int qoff[8];
#pragma unroll
                for (int p = 0; p < 8; ++p) {
                    const int g32 = (int)(row0 + rsub + RSTEP * (pb + p));
                    const int batch = a.tile_in_batch ? tile_batch : g32 / a.rows_per_batch;
                    const int qrow = a.q_shift >= 0 ? g32 >> a.q_shift : g32 / a.q_ns;
                    const int gidx = gi[pb + p];
                    src[p] = gidx >= 0 ? ((long long)batch * a.n_src + gidx) * a.ldp : -1;
                    qoff[p] = gidx >= 0 ? qrow * a.ldq : 0;
                }
                for (int kc = kc_lo; kc < kc_hi; ++kc) {
                    const int k = kc * 64 + 4 * jv;
                    const bool k_ok = k < a.c1;
                    float4 pv[8], qv[8];
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        const bool ok = k_ok && src[p] >= 0;
                        pv[p] = ok ? __ldg(reinterpret_cast<const float4 *>(a.P + src[p] + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
                        qv[p] = ok ? __ldg(reinterpret_cast<const float4 *>(a.Q + qoff[p] + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int p = 0; p < 8; ++p) {
                        const int rl = rsub + RSTEP * (pb + p);
                        const float x0 = fmaxf(pv[p].x - qv[p].x, 0.f), x1 = fmaxf(pv[p].y - qv[p].y, 0.f);
                        const float x2 = fmaxf(pv[p].z - qv[p].z, 0.f), x3 = fmaxf(pv[p].w - qv[p].w, 0.f);
                        if (NPASS == 2) {   // k 4 jv .. 4 jv + 3 of the atom: image jv / 8, 16-byte unit jv % 8
                            const uint32_t toff = (jv >> 3) * (k1 * ATOM) + kc * ATOM + rl * 128 + (((jv & 7) ^ (rl & 7)) << 4);
                            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(A_hi + toff), "r"(tf32_rna_bits((x0))),
                                         "r"(tf32_rna_bits((x1))), "r"(tf32_rna_bits((x2))), "r"(tf32_rna_bits((x3))));
                            continue;
                        }
                        const uint32_t off = kc * ATOM + rl * 128 + (((jv >> 1) ^ (rl & 7)) << 4) + ((jv & 1) << 3);
                        const __nv_bfloat162 h0 = __floats2bfloat162_rn(x0, x1), h1 = __floats2bfloat162_rn(x2, x3);
                        asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(A_hi + off), "r"(*reinterpret_cast<const uint32_t *>(&h0)),
                                     "r"(*reinterpret_cast<const uint32_t *>(&h1)));
                        if (NPASS == 3) {
                            const float2 f0 = __bfloat1622float2(h0), f1 = __bfloat1622float2(h1);
                            const __nv_bfloat162 l0 = __floats2bfloat162_rn(x0 - f0.x, x1 - f0.y);
                            const __nv_bfloat162 l1 = __floats2bfloat162_rn(x2 - f1.x, x3 - f1.y);
                            asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(A_lo + off), "r"(*reinterpret_cast<const uint32_t *>(&l0)),
                                         "r"(*reinterpret_cast<const uint32_t *>(&l1)));
                        }
                    }
                }
            }
            if (last) {
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(a_ready);
            }
        };
        long long cy[7] = {0, 0, 0, 0, 0, 0, 0};
        long long tt = clock64();
        auto lap = [&](int i) { const long long n = clock64(); cy[i] += n - tt; tt = n; };
        uint32_t ph_d1 = 0, ph_d2 = 0;
        // the gather of the next tile is spread over the passes of the second GEMM (one part before each pooling pass),
        // so that the tensor pipe always has the next pass to run while the workers gather
        const int nparts = np2 < k1 ? np2 : k1;
        request(0);
        gather(0, 0, k1, true);
        lap(0);
        for (int t = 0; t < my_tiles; ++t) {
            const long long row0 = ((long long)blockIdx.x + (long long)t * gridDim.x) * BM;
            request(t + 1);
            lap(1);
            // ---- hidden layer: H = relu(D + b1) -> TMEM A operand of the second GEMM (zero beyond c2, up to whole k-atoms) ----
            for (int p = 0; p < np1; ++p) {
                mbar_wait(d1bar, ph_d1); ph_d1 ^= 1;
                tc_fence_after();
                lap(2);
                const int g_lo = p * DN / 32, g_hi = min(2 * k2, (p + 1) * DN / 32);
                for (int g = g_lo + half; g < g_hi; g += HALVES) {
                    if (NPASS == 2) {   // tf32: H column k = n, 32 columns per group
                        uint32_t r[32];
                        if (g * 32 < bn1) {
                            tmem_ld32(lane_addr + dcol + (g * 32 - p * DN), r);
#pragma unroll
                            for (int j = 0; j < 32; ++j) {
                                const int n = g * 32 + j;
                                r[j] = n < a.c2 ? tf32_rna_bits((fmaxf(__uint_as_float(r[j]) + b1p[n], 0.f))) : 0u;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 32; ++j) r[j] = 0u;
                        }
                        tmem_st32(lane_addr + (uint32_t)(g * 32), r);
                        continue;
                    }
                    uint32_t hi[16], lo[16];
                    if (g * 32 < bn1) {
                        uint32_t r[32];
                        tmem_ld32(lane_addr + dcol + (g * 32 - p * DN), r);
#pragma unroll
                        for (int j4 = 0; j4 < 8; ++j4) {
                            const int n0 = g * 32 + j4 * 4;
                            float v[4];
#pragma unroll
                            for (int j = 0; j < 4; ++j) v[j] = n0 + j < a.c2 ? fmaxf(__uint_as_float(r[j4 * 4 + j]) + b1p[n0 + j], 0.f) : 0.f;
                            const __nv_bfloat162 p0 = __floats2bfloat162_rn(v[0], v[1]), p1 = __floats2bfloat162_rn(v[2], v[3]);
                            hi[j4 * 2 + 0] = *reinterpret_cast<const uint32_t *>(&p0);
                            hi[j4 * 2 + 1] = *reinterpret_cast<const uint32_t *>(&p1);
                            if (NPASS == 3) {
                                const float2 f0 = __bfloat1622float2(p0), f1 = __bfloat1622float2(p1);
                                const __nv_bfloat162 l0 = __floats2bfloat162_rn(v[0] - f0.x, v[1] - f0.y), l1 = __floats2bfloat162_rn(v[2] - f1.x, v[3] - f1.y);
                                lo[j4 * 2 + 0] = *reinterpret_cast<const uint32_t *>(&l0);
                                lo[j4 * 2 + 1] = *reinterpret_cast<const uint32_t *>(&l1);
                            }
                        }
                    } else {   // padding columns of the last k-atom beyond the accumulator width: zeros
#pragma unroll
                        for (int j = 0; j < 16; ++j) { hi[j] = 0u; lo[j] = 0u; }
                    }
                    tmem_st16(lane_addr + (uint32_t)(g * 16), hi);                       // H hi: column n / 2
                    if (NPASS == 3) tmem_st16(lane_addr + (uint32_t)(k2 * 32 + g * 16), lo);
                }
                tmem_st_wait();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(e1_done);
                lap(3);
            }
            // ---- output layer + max-pool over the pool_ns rows of each group; before each pooling pass a part of the NEXT
            // tile is gathered while the tensor pipe runs that pass of the second GEMM (GEMM 1 of this tile has retired) ----
            const long long grow = row0 + row;
            const bool row_ok = grow < a.R;
            for (int q = 0; q < np2; ++q) {
                if (t + 1 < my_tiles && q < nparts) gather(t + 1, q * k1 / nparts, (q + 1) * k1 / nparts, q == nparts - 1);
                lap(0);
                mbar_wait(d2bar, ph_d2); ph_d2 ^= 1;
                tc_fence_after();
                lap(4);
                const int g_lo = q * DN / 32, g_hi = min((a.c3 + 31) / 32, (q + 1) * DN / 32);
                for (int g = g_lo + half; g < g_hi; g += HALVES) {
                    uint32_t r[32];
                    tmem_ld32(lane_addr + dcol + (g * 32 - q * DN), r);
#ifdef GP_SAF_PROBE
                    { const long long n = clock64(); cy[6] += n - tt; }
#endif
                    if (ns == 32) pool_block<32>(r, row_ok, lane, row0 + 32 * quarter, a.R, g * 32, a.c3, b2p, a.pooled, a.ld_pooled, vec_ok);
                    else if (ns == 16) pool_block<16>(r, row_ok, lane, row0 + 32 * quarter, a.R, g * 32, a.c3, b2p, a.pooled, a.ld_pooled, vec_ok);
                    else pool_block<8>(r, row_ok, lane, row0 + 32 * quarter, a.R, g * 32, a.c3, b2p, a.pooled, a.ld_pooled, vec_ok);
                }
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(p_done);
                lap(5);
            }
        }
#ifdef GP_SAF_PROBE
        if (blockIdx.x == 0 && tid == 64)
            printf("saf c=(%d,%d,%d) ns=%d tiles=%d per tile: gather %lld locate %lld wait_d0 %lld hidden %lld wait_d1 %lld pool %lld (cumulative to each ldtm %lld)\n", a.c1, a.c2,
                   a.c3, a.pool_ns, my_tiles, cy[0] / my_tiles, cy[1] / my_tiles, cy[2] / my_tiles, cy[3] / my_tiles, cy[4] / my_tiles, cy[5] / my_tiles, cy[6] / my_tiles);
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem, (uint32_t)a.tmem_cols);
}

// TMEM / shared-memory plan of a shape.  Returns false when it does not fit (the caller reports GP_ERR_UNSUPPORTED).
template <int NPASS>
static bool plan(Args &a, bool two_per_sm, size_t smem_budget) {
    constexpr int IM = Cfg<NPASS>::IMAGES;
    const int k2 = atoms_of(a.c2);
    a.tmem_cols = two_per_sm ? 256 : 512;
    a.hcols = k2 * 32 * IM;
    const int avail = a.tmem_cols - a.hcols;
    if (avail < 128) return false;
    a.dn = avail >= 256 ? 256 : 128;
    for (int bias_smem = 1; bias_smem >= 0; --bias_smem) {
        a.bias_smem = bias_smem;
        const size_t fixed = Layout<NPASS>(a.c1, 0, bias_smem).total();
        if (fixed + 2 * (size_t)SLOT * IM > smem_budget) continue;
        const int nst = (int)((smem_budget - fixed) / SLOT);
        a.nst = nst > MAX_NST ? MAX_NST : nst;
        return true;
    }
    return false;
}

template <int NPASS>
static int launch(Args a, cudaStream_t st) {
    a.tile_in_batch = a.rows_per_batch % BM == 0;
    a.q_shift = -1;
    for (int sh = 0; sh < 31; ++sh)
        if ((1 << sh) == a.q_ns) a.q_shift = sh;
    // two 192-thread CTAs per SM when one of them fits in half of the shared memory and 256 TMEM columns with both
    // GEMMs in a single accumulator pass (the narrow levels: their tiles are gather / pool bound, a second CTA doubles
    // the warps that hide those latencies)
    Args a2 = a;
    if (plan<NPASS>(a2, true, 113 * 1024) && round16(a.c2) <= a2.dn && round16(a.c3) <= a2.dn) {
        const Layout<NPASS> L2(a2.c1, a2.nst, a2.bias_smem);
        auto kern = sa_mlp2_kernel<NPASS, 4>;
        GP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        GP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        const int cap = 2 * num_sms();
        kern<<<a2.ntiles < cap ? a2.ntiles : cap, 6 * 32, L2.total(), st>>>(a2);
        GP_CHECK_LAUNCH("gp_sa_mlp2_fused");
        return GP_OK;
    }
    if (!plan<NPASS>(a, false, 227 * 1024)) {
        set_error("gp_sa_mlp2_fused: widths (%d, %d, %d) do not fit tensor / shared memory", a.c1, a.c2, a.c3);
        return GP_ERR_UNSUPPORTED;
    }
    const Layout<NPASS> L(a.c1, a.nst, a.bias_smem);
    auto kern = sa_mlp2_kernel<NPASS, 8>;
    GP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    const int grid = a.ntiles < num_sms() ? a.ntiles : num_sms();
    kern<<<grid, 10 * 32, L.total(), st>>>(a);
    GP_CHECK_LAUNCH("gp_sa_mlp2_fused");
    return GP_OK;
}

}  // namespace saf
}  // namespace gp

using namespace gp;

static int launch_npass(const saf::Args &a, int npass, cudaStream_t st) {
    return npass == 3 ? saf::launch<3>(a, st) : npass == 2 ? saf::launch<2>(a, st) : saf::launch<1>(a, st);
}

extern "C" int gp_sa_mlp2_fused(const float *P, int n_src, int ldp, const int32_t *gidx, long long R, int rows_per_batch,
                                const float *Q, int ldq, int q_ns, const void *packed1, const float *bias1, int c1, int c2,
                                const void *packed2, const float *bias2, int c3, int npass, int pool_ns, float *pooled,
                                int ld_pooled, gp_stream_t s) {
    GP_REQUIRE(R >= 0 && npass >= 1 && npass <= 3, "gp_sa_mlp2_fused: bad arguments (npass must be 1, 2 or 3)");
    if (R == 0) return GP_OK;
    GP_REQUIRE(P && gidx && Q && packed1 && bias1 && packed2 && bias2 && pooled, "gp_sa_mlp2_fused: null pointer");
    GP_REQUIRE(c1 >= 4 && c1 <= 256 && (c1 & 3) == 0 && c2 >= 1 && c2 <= 384 && c3 >= 1 && c3 <= 512,
               "gp_sa_mlp2_fused: widths must satisfy c1 %% 4 == 0, c1 <= 256, c2 <= 384 and c3 <= 512 (got %d, %d, %d)", c1, c2, c3);
    GP_REQUIRE(ldp >= c1 && (ldp & 3) == 0 && ((uintptr_t)P & 15) == 0 && ldq >= c1 && (ldq & 3) == 0 && ((uintptr_t)Q & 15) == 0,
               "gp_sa_mlp2_fused: P / Q rows must be 16-byte aligned and cover c1");
    GP_REQUIRE(((uintptr_t)packed1 & 15) == 0 && ((uintptr_t)packed2 & 15) == 0, "gp_sa_mlp2_fused: packed weights must be 16-byte aligned");
    GP_REQUIRE(rows_per_batch >= 1 && n_src >= 1 && q_ns >= 1, "gp_sa_mlp2_fused: bad gather geometry");
    GP_REQUIRE((pool_ns == 8 || pool_ns == 16 || pool_ns == 32) && R % pool_ns == 0 && ld_pooled >= c3,
               "gp_sa_mlp2_fused: pool_ns must be 8, 16 or 32 and divide R");
    GP_REQUIRE(R < 2147483647LL && (R / q_ns + 1) * (long long)ldq < 2147483647LL, "gp_sa_mlp2_fused: too many rows");
    saf::Args a;
    a.P = P; a.n_src = n_src; a.ldp = ldp; a.gidx = gidx; a.R = R; a.rows_per_batch = rows_per_batch;
    a.Q = Q; a.ldq = ldq; a.q_ns = q_ns;
    a.W1p = (const uint8_t *)packed1; a.b1 = bias1; a.c1 = c1; a.c2 = c2;
    a.W2p = (const uint8_t *)packed2; a.b2 = bias2; a.c3 = c3;
    a.pool_ns = pool_ns; a.pooled = pooled; a.ld_pooled = ld_pooled;
    a.ntiles = (int)((R + saf::BM - 1) / saf::BM);
    a.xyz = nullptr; a.centres = nullptr;
    return launch_npass(a, npass, as_stream(s));
}

extern "C" int gp_sa_mlp2_fused_xyz(const float *xyz, const float *centres, int n_src, const int32_t *gidx, long long R,
                                    int rows_per_batch, int q_ns, const float *host_W0, const float *host_b0, const void *packed1,
                                    const float *bias1, int c1, int c2, const void *packed2, const float *bias2, int c3, int npass,
                                    int pool_ns, float *pooled, int ld_pooled, gp_stream_t s) {
    GP_REQUIRE(R >= 0 && npass >= 1 && npass <= 3, "gp_sa_mlp2_fused_xyz: bad arguments (npass must be 1, 2 or 3)");
    if (R == 0) return GP_OK;
    GP_REQUIRE(xyz && centres && gidx && host_W0 && host_b0 && packed1 && bias1 && packed2 && bias2 && pooled, "gp_sa_mlp2_fused_xyz: null pointer");
    GP_REQUIRE((c1 == 16 || c1 == 32) && c2 >= 1 && c2 <= 384 && c3 >= 1 && c3 <= 512,
               "gp_sa_mlp2_fused_xyz: c1 must be 16 or 32, c2 <= 384 and c3 <= 512 (got %d, %d, %d)", c1, c2, c3);
    GP_REQUIRE(((uintptr_t)packed1 & 15) == 0 && ((uintptr_t)packed2 & 15) == 0, "gp_sa_mlp2_fused_xyz: packed weights must be 16-byte aligned");
    GP_REQUIRE(rows_per_batch >= 1 && n_src >= 1 && q_ns >= 1, "gp_sa_mlp2_fused_xyz: bad gather geometry");
    GP_REQUIRE((pool_ns == 8 || pool_ns == 16 || pool_ns == 32) && R % pool_ns == 0 && ld_pooled >= c3,
               "gp_sa_mlp2_fused_xyz: pool_ns must be 8, 16 or 32 and divide R");
    GP_REQUIRE(R < 2147483647LL, "gp_sa_mlp2_fused_xyz: too many rows");
    saf::Args a;
    a.P = nullptr; a.n_src = n_src; a.ldp = 0; a.gidx = gidx; a.R = R; a.rows_per_batch = rows_per_batch;
    a.Q = nullptr; a.ldq = 0; a.q_ns = q_ns;
    a.W1p = (const uint8_t *)packed1; a.b1 = bias1; a.c1 = c1; a.c2 = c2;
    a.W2p = (const uint8_t *)packed2; a.b2 = bias2; a.c3 = c3;
    a.pool_ns = pool_ns; a.pooled = pooled; a.ld_pooled = ld_pooled;
    a.ntiles = (int)((R + saf::BM - 1) / saf::BM);
    a.xyz = xyz; a.centres = centres;
    for (int k = 0; k < 64; ++k) {
        a.b0c[k] = k < c1 ? host_b0[k] : 0.f;
        for (int d = 0; d < 3; ++d) a.w0c[k * 3 + d] = k < c1 ? host_W0[k * 3 + d] : 0.f;
    }
    return launch_npass(a, npass, as_stream(s));
}
