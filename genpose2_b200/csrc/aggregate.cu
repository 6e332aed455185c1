// Energy-ranked outlier rejection + quaternion averaging + DBSCAN mode selection, one warp per
// object, and the ScaleNet bbox head.  Replaces the Python / sklearn / cuSOLVER host loop of
// runners/evaluation_single.py:179-215 (one D2H + sklearn call per object) with segmented
// reductions that never leave the device.
// Energies are ranked like torch.sort(descending=True, stable=True) (NaN above +inf, ties by index), so an object whose
// retained set holds a NaN pose comes out NaN in rows 0-2 with labels -1, and no other object changes.
#include "common.cuh"

namespace gp {

constexpr int AG_WARPS = 4;     // objects per block
constexpr int AG_MAXR = 64;     // hypotheses per object
constexpr int AG_MAXK = 32;     // retained hypotheses (DBSCAN neighbourhoods are 32-bit masks)

struct AggSmem {
    unsigned e[AG_MAXR][2];      // rank_key of the energies
    int order[2][AG_MAXR];       // rank -> hypothesis, per energy channel
    double q[AG_MAXR][4];        // retained quaternions (wxyz); more than AG_MAXK only without clustering
    double D[AG_MAXK][AG_MAXK];  // 1 - <qi,qj>^2
    unsigned nbr[AG_MAXK];
};

// rotation_6d_to_matrix(.).permute(0,2,1) then matrix_to_quaternion
// (rotation_conversions.py:556-577, 102-161; misc.py:148-149), float64.
__device__ void rot6d_to_quat(const double *d6, double *q) {
    const double eps = 1e-12;
    double n1 = sqrt(d6[0] * d6[0] + d6[1] * d6[1] + d6[2] * d6[2]);
    n1 = n1 > eps ? n1 : eps;
    const double b1[3] = {d6[0] / n1, d6[1] / n1, d6[2] / n1};
    const double dt = b1[0] * d6[3] + b1[1] * d6[4] + b1[2] * d6[5];
    double b2[3] = {d6[3] - dt * b1[0], d6[4] - dt * b1[1], d6[5] - dt * b1[2]};
    double n2 = sqrt(b2[0] * b2[0] + b2[1] * b2[1] + b2[2] * b2[2]);
    n2 = n2 > eps ? n2 : eps;
    b2[0] /= n2; b2[1] /= n2; b2[2] /= n2;
    const double b3[3] = {b1[1] * b2[2] - b1[2] * b2[1], b1[2] * b2[0] - b1[0] * b2[2], b1[0] * b2[1] - b1[1] * b2[0]};
    // columns of the rotation matrix are b1, b2, b3
    const double m00 = b1[0], m10 = b1[1], m20 = b1[2];
    const double m01 = b2[0], m11 = b2[1], m21 = b2[2];
    const double m02 = b3[0], m12 = b3[1], m22 = b3[2];
    double x[4] = {1.0 + m00 + m11 + m22, 1.0 + m00 - m11 - m22, 1.0 - m00 + m11 - m22, 1.0 - m00 - m11 + m22};
    double qa[4];
    int best = 0;
    for (int i = 0; i < 4; ++i) {
        qa[i] = x[i] > 0 ? sqrt(x[i]) : 0.0;
        if (qa[i] > qa[best]) best = i;  // argmax, first occurrence
    }
    double cand[4];
    switch (best) {
        case 0: cand[0] = qa[0] * qa[0]; cand[1] = m21 - m12; cand[2] = m02 - m20; cand[3] = m10 - m01; break;
        case 1: cand[0] = m21 - m12; cand[1] = qa[1] * qa[1]; cand[2] = m10 + m01; cand[3] = m02 + m20; break;
        case 2: cand[0] = m02 - m20; cand[1] = m10 + m01; cand[2] = qa[2] * qa[2]; cand[3] = m12 + m21; break;
        default: cand[0] = m10 - m01; cand[1] = m20 + m02; cand[2] = m21 + m12; cand[3] = qa[3] * qa[3]; break;
    }
    const double den = 2.0 * (qa[best] > 0.1 ? qa[best] : 0.1);
    for (int i = 0; i < 4; ++i) q[i] = cand[i] / den;
}

// principal eigenvector of the symmetric 4x4 matrix A (cyclic Jacobi, float64), oriented w > 0
// like average_quaternion_batch (misc.py:315-317).
__device__ void top_eigvec4(double A[4][4], double *out) {
    double V[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
    for (int sweep = 0; sweep < 32; ++sweep) {
        double off = 0.0, diag = 0.0;
        for (int i = 0; i < 4; ++i) {
            diag += A[i][i] * A[i][i];
            for (int j = i + 1; j < 4; ++j) off += A[i][j] * A[i][j];
        }
        if (off <= 1e-34 * diag || off == 0.0) break;
        for (int p = 0; p < 3; ++p)
            for (int q = p + 1; q < 4; ++q) {
                const double apq = A[p][q];
                if (apq == 0.0) continue;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
                const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < 4; ++k) {  // A <- A J
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - s * akq;
                    A[k][q] = s * akp + c * akq;
                }
                for (int k = 0; k < 4; ++k) {  // A <- J^T A
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - s * aqk;
                    A[q][k] = s * apk + c * aqk;
                }
                for (int k = 0; k < 4; ++k) {
                    const double vkp = V[k][p], vkq = V[k][q];
                    V[k][p] = c * vkp - s * vkq;
                    V[k][q] = s * vkp + c * vkq;
                }
            }
    }
    int best = 0;
    for (int i = 1; i < 4; ++i)
        if (A[i][i] > A[best][best]) best = i;
    const double sgn = V[0][best] > 0 ? 1.0 : -1.0;
    for (int k = 0; k < 4; ++k) out[k] = sgn * V[k][best];
}

// A = sum over the members in `mask` of (oriented q)(oriented q)^T; scale is irrelevant to the
// eigenvector, members are oriented to w > 0 exactly like ((Q[...,0:1] > 0) - 0.5) * 2 * Q.
__device__ void average_quat(const double (*q)[4], unsigned long long mask, double *out) {
    double A[4][4] = {};
    for (int i = 0; i < AG_MAXR; ++i) {
        if (!((mask >> i) & 1ull)) continue;
        const double sg = q[i][0] > 0 ? 1.0 : -1.0;
        double v[4] = {sg * q[i][0], sg * q[i][1], sg * q[i][2], sg * q[i][3]};
        for (int a = 0; a < 4; ++a)
            for (int b = 0; b < 4; ++b) A[a][b] += v[a] * v[b];
    }
    top_eigvec4(A, out);
}

// rank key of an energy: descending unsigned order of the keys is torch.sort(descending=True)'s order -- every NaN
// (any payload) one key above +inf, -0 the key of +0 -- so with ties broken by index the ranks are a permutation
// whatever the energies are.  Keys are made once per energy; the rank loop compares integers.
__device__ __forceinline__ unsigned rank_key(float e) {
    const unsigned u = e != e ? 0x7fc00000u : (e == 0.f ? 0u : __float_as_uint(e));
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__global__ void __launch_bounds__(AG_WARPS * 32)
aggregate_kernel(const double *__restrict__ poses, const float *__restrict__ energy, int B, int R, int retain,
                 int clustering, double eps, int min_samples, float *__restrict__ pose_out,
                 int *__restrict__ labels_out, double *__restrict__ sorted_out) {
    __shared__ AggSmem sm[AG_WARPS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * AG_WARPS + warp;
    if (b >= B) return;
    AggSmem &S = sm[warp];
    const double *P = poses + (size_t)b * R * 9;

    for (int i = lane; i < R * 2; i += 32) S.e[i >> 1][i & 1] = rank_key(energy[(size_t)b * R * 2 + i]);
    __syncwarp();
    // descending stable rank per channel (torch.sort(energy, descending=True, dim=1), reward.py:145)
    for (int i = lane; i < R; i += 32) {
        for (int ch = 0; ch < 2; ++ch) {
            const unsigned ei = S.e[i][ch];
            int rank = 0;
            for (int j = 0; j < R; ++j) {
                const unsigned ej = S.e[j][ch];
                rank += (ej > ei) || (ej == ei && j < i);
            }
            S.order[ch][rank] = i;
        }
    }
    __syncwarp();
    if (sorted_out) {
        for (int i = lane; i < R * 9; i += 32) {
            const int r = i / 9, c = i - 9 * r;
            sorted_out[(size_t)b * R * 9 + i] = P[(size_t)S.order[c < 6 ? 0 : 1][r] * 9 + c];
        }
    }
    // retained quaternions
    for (int i = lane; i < retain; i += 32) {
        double d6[6];
        for (int c = 0; c < 6; ++c) d6[c] = P[(size_t)S.order[0][i] * 9 + c];
        rot6d_to_quat(d6, S.q[i]);
    }
    __syncwarp();
    const unsigned long long all = retain >= 64 ? ~0ull : ((1ull << retain) - 1ull);
    unsigned long long member = all;
    if (clustering) {
        for (int i = lane; i < retain * retain; i += 32) {
            const int r = i / retain, c = i - r * retain;
            const double dot = S.q[r][0] * S.q[c][0] + S.q[r][1] * S.q[c][1] + S.q[r][2] * S.q[c][2] + S.q[r][3] * S.q[c][3];
            S.D[r][c] = 1.0 - dot * dot;
        }
        __syncwarp();
        // DBSCAN on the ROWS of D as feature vectors, Euclidean, <= eps (SURVEY.md Appendix A)
        for (int i = lane; i < retain; i += 32) {
            unsigned m = 0;
            for (int j = 0; j < retain; ++j) {
                double s = 0.0;
                for (int k = 0; k < retain; ++k) {
                    const double d = S.D[i][k] - S.D[j][k];
                    s += d * d;
                }
                if (sqrt(s) <= eps) m |= 1u << j;
            }
            S.nbr[i] = m;
        }
        __syncwarp();
    }
    if (lane == 0) {
        int labels[AG_MAXR];
        for (int i = 0; i < retain; ++i) labels[i] = -1;
        if (clustering) {
            unsigned core = 0, labeled = 0;
            for (int i = 0; i < retain; ++i)
                if (__popc(S.nbr[i]) >= min_samples) core |= 1u << i;
            int label = 0, best_label = -1, best_count = 0;
            unsigned best_members = 0;
            for (int i = 0; i < retain; ++i) {
                if (((labeled >> i) & 1u) || !((core >> i) & 1u)) continue;
                unsigned frontier = 1u << i, members = 0;
                while (frontier) {
                    const int j = __ffs(frontier) - 1;
                    frontier &= ~(1u << j);
                    if ((labeled >> j) & 1u) continue;
                    labeled |= 1u << j;
                    members |= 1u << j;
                    labels[j] = label;
                    if ((core >> j) & 1u) frontier |= S.nbr[j] & ~labeled;
                }
                const int cnt = __popc(members);
                if (cnt > best_count) {  // np.argmax(np.bincount(...)): first maximum
                    best_count = cnt;
                    best_label = label;
                    best_members = members;
                }
                ++label;
            }
            if (best_label >= 0) member = best_members;
        }
        if (labels_out)
            for (int i = 0; i < retain; ++i) labels_out[(size_t)b * retain + i] = labels[i];
        double qavg[4];
        average_quat(S.q, member, qavg);
        // quaternion_to_matrix (rotation_conversions.py:41-70)
        const double r = qavg[0], i = qavg[1], j = qavg[2], k = qavg[3];
        const double two_s = 2.0 / (r * r + i * i + j * j + k * k);
        double t[3] = {0, 0, 0};
        for (int n = 0; n < retain; ++n)
            for (int c = 0; c < 3; ++c) t[c] += P[(size_t)S.order[1][n] * 9 + 6 + c];
        float *o = pose_out + (size_t)b * 16;
        o[0] = (float)(1 - two_s * (j * j + k * k)); o[1] = (float)(two_s * (i * j - k * r)); o[2] = (float)(two_s * (i * k + j * r));
        o[4] = (float)(two_s * (i * j + k * r)); o[5] = (float)(1 - two_s * (i * i + k * k)); o[6] = (float)(two_s * (j * k - i * r));
        o[8] = (float)(two_s * (i * k - j * r)); o[9] = (float)(two_s * (j * k + i * r)); o[10] = (float)(1 - two_s * (i * i + j * j));
        o[3] = (float)(t[0] / retain); o[7] = (float)(t[1] / retain); o[11] = (float)(t[2] / retain);
        o[12] = 0.f; o[13] = 0.f; o[14] = 0.f; o[15] = 1.f;
    }
}

// ------------------------------------------------------------------------------------------
// ScaleNet (networks/scalenet.py:33-49) + encode_axes (utils/genpose_utils.py:8-18)
// OB objects per block share every weight row they stream.
// ------------------------------------------------------------------------------------------
template <int OB>
struct ScaleSmem {
    float in0[OB][192];    // 180 used: [sin(90) | cos(90)]
    float h0[OB][256];
    float tot[OB][1280];   // [pts_feat(1024) | axes_feat(256)]  (scalenet.py:46)
    float h1[OB][256];
};

// out[o][n] = act(b[n] + sum_k W[n][k] in[o][k]); one warp per output n, every lane takes 4 consecutive k per step
// (16-byte loads: the weight row streams from L2 once per CTA).  A warp works on NB outputs at a time -- all their weight
// loads are in flight together, so a layer costs NOUT / (8 NB) L2 round trips per warp instead of NOUT / 8 (the kernel is
// bound by that latency chain: 64 CTAs, one object each at C2).  K % 4 == 0.
template <int OB, int K, int LD, bool RELU>
__device__ __forceinline__ void dense_rows(const float *__restrict__ W, const float *__restrict__ bias, int NOUT,
                                           const float *in, float *out, int out_ld) {
    static_assert(K % 4 == 0 && LD % 4 == 0, "16-byte rows");
    constexpr int STEPS = (K / 4 + 31) / 32;
    constexpr int NB = STEPS * OB <= 2 ? 8 : (STEPS * OB <= 4 ? 4 : (STEPS <= 12 && OB <= 2 ? 2 : 1));
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
    for (int n0 = warp * NB; n0 < NOUT; n0 += nw * NB) {
        float4 wv[NB][STEPS];
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            const int n = n0 + j < NOUT ? n0 + j : NOUT - 1;
            const float4 *w = reinterpret_cast<const float4 *>(W + (size_t)n * K);
#pragma unroll
            for (int i = 0; i < STEPS; ++i) {
                const int k4 = lane + 32 * i;
                wv[j][i] = k4 < K / 4 ? __ldg(w + k4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        float acc[NB][OB];
#pragma unroll
        for (int j = 0; j < NB; ++j)
#pragma unroll
            for (int o = 0; o < OB; ++o) acc[j][o] = 0.f;
#pragma unroll
        for (int i = 0; i < STEPS; ++i) {
            const int k4 = lane + 32 * i;
            if (k4 < K / 4) {
#pragma unroll
                for (int o = 0; o < OB; ++o) {
                    const float4 x = *reinterpret_cast<const float4 *>(in + o * LD + 4 * k4);
#pragma unroll
                    for (int j = 0; j < NB; ++j)
                        acc[j][o] = fmaf(x.x, wv[j][i].x, fmaf(x.y, wv[j][i].y, fmaf(x.z, wv[j][i].z, fmaf(x.w, wv[j][i].w, acc[j][o]))));
                }
            }
        }
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            const int n = n0 + j;
            if (n >= NOUT) break;
            const float bv = __ldg(bias + n);
#pragma unroll
            for (int o = 0; o < OB; ++o) {
                float v = acc[j][o];
#pragma unroll
                for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
                v += bv;
                if (lane == 0) out[o * out_ld + n] = RELU && v == v ? fmaxf(v, 0.f) : v;   // NaN passes, like torch.relu
            }
        }
    }
}

template <int OB>
__global__ void __launch_bounds__(256)
scalenet_kernel(gp_scalenet_params p, const float *__restrict__ axes, int bstride, int rstride,
                const float *__restrict__ feat, int B, float *__restrict__ length) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    ScaleSmem<OB> &S = *reinterpret_cast<ScaleSmem<OB> *>(smem_raw);
    const int b0 = blockIdx.x * OB, tid = threadIdx.x;
    for (int i = tid; i < OB * 90; i += 256) {
        const int o = i / 90, e = i - 90 * o;       // e = elem*10 + k, elem = row*3 + col
        const int elem = e / 10, k = e - 10 * elem;
        float a = 0.f;
        if (b0 + o < B) a = axes[(size_t)(b0 + o) * bstride + (elem / 3) * rstride + (elem % 3)];
        const float arg = __fmul_rn((float)(1 << k), a);
        float sn, cs;
        sincosf(arg, &sn, &cs);
        S.in0[o][e] = sn;
        S.in0[o][90 + e] = cs;
    }
    for (int i = tid; i < OB * 1024; i += 256) {
        const int o = i >> 10, c = i & 1023;
        S.tot[o][c] = (b0 + o < B) ? feat[(size_t)(b0 + o) * 1024 + c] : 0.f;
    }
    __syncthreads();
    dense_rows<OB, 180, 192, true>(p.axes_w0, p.axes_b0, 256, &S.in0[0][0], &S.h0[0][0], 256);
    __syncthreads();
    dense_rows<OB, 256, 256, true>(p.axes_w1, p.axes_b1, 256, &S.h0[0][0], &S.tot[0][1024], 1280);
    __syncthreads();
    dense_rows<OB, 1280, 1280, true>(p.tail_w0, p.tail_b0, 256, &S.tot[0][0], &S.h1[0][0], 256);
    __syncthreads();
    float *out_s = &S.h0[0][0];  // reuse: [OB][256], 3 used
    dense_rows<OB, 256, 256, false>(p.tail_w1, p.tail_b1, 3, &S.h1[0][0], out_s, 256);
    __syncthreads();
    for (int i = tid; i < OB * 3; i += 256) {
        const int o = i / 3, c = i - 3 * o;
        if (b0 + o < B) length[(size_t)(b0 + o) * 3 + c] = out_s[o * 256 + c];
    }
}

// pred_pose_q_wxyz of PoseNet.pred_func (posenet_agent.py:547-559): [x-axis(3) y-axis(3) t(3)] f64 -> [q_wxyz(4) t(3)]
__global__ void pose_to_quat_kernel(const double *__restrict__ poses, int N, double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= N) return;
    double v[9], q[4];
#pragma unroll
    for (int c = 0; c < 9; ++c) v[c] = poses[(size_t)i * 9 + c];
    rot6d_to_quat(v, q);
#pragma unroll
    for (int c = 0; c < 4; ++c) out[(size_t)i * 7 + c] = q[c];
#pragma unroll
    for (int c = 0; c < 3; ++c) out[(size_t)i * 7 + 4 + c] = v[6 + c];
}

}  // namespace gp

using namespace gp;

extern "C" int gp_pose_to_quat(const double *poses, int N, double *out, gp_stream_t s) {
    GP_REQUIRE(poses && out && N >= 0, "gp_pose_to_quat: bad arguments");
    if (N == 0) return GP_OK;
    pose_to_quat_kernel<<<(N + 127) / 128, 128, 0, as_stream(s)>>>(poses, N, out);
    GP_CHECK_LAUNCH("gp_pose_to_quat");
    return GP_OK;
}

extern "C" int gp_aggregate(const double *poses, const float *energy, int B, int R, int retain, int clustering,
                            double clustering_eps, int min_samples, float *pose_out, int32_t *labels_out,
                            double *sorted_out, gp_stream_t s) {
    GP_REQUIRE(poses && energy && pose_out, "gp_aggregate: null pointer");
    GP_REQUIRE(B >= 0 && R >= 1 && R <= AG_MAXR, "gp_aggregate: R=%d must be in [1,%d]", R, AG_MAXR);
    GP_REQUIRE(retain >= 1 && retain <= (clustering ? AG_MAXK : AG_MAXR) && retain <= R,
               "gp_aggregate: retain=%d must be in [1,min(R,%d)] (%d without clustering)", retain, AG_MAXK, AG_MAXR);
    if (B == 0) return GP_OK;
    aggregate_kernel<<<(B + AG_WARPS - 1) / AG_WARPS, AG_WARPS * 32, 0, as_stream(s)>>>(
        poses, energy, B, R, retain, clustering, clustering_eps, min_samples, pose_out, labels_out, sorted_out);
    GP_CHECK_LAUNCH("gp_aggregate");
    return GP_OK;
}

template <int OB>
static int launch_scalenet(const gp_scalenet_params *p, const float *axes, int bs, int rs, const float *feat, int B,
                           float *length, cudaStream_t st) {
    const size_t smem = sizeof(ScaleSmem<OB>);
    auto kern = scalenet_kernel<OB>;
    if (smem > 48 * 1024) GP_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<(B + OB - 1) / OB, 256, smem, st>>>(*p, axes, bs, rs, feat, B, length);
    GP_CHECK_LAUNCH("gp_scalenet");
    return GP_OK;
}

extern "C" int gp_scalenet(const gp_scalenet_params *p, const float *axes, int axes_batch_stride, int axes_row_stride,
                           const float *pts_feat, int B, float *length, gp_stream_t s) {
    GP_REQUIRE(p && axes && pts_feat && length, "gp_scalenet: null pointer");
    GP_REQUIRE(p->axes_w0 && p->axes_b0 && p->axes_w1 && p->axes_b1 && p->tail_w0 && p->tail_b0 && p->tail_w1 && p->tail_b1,
               "gp_scalenet: null parameter");
    GP_REQUIRE(B >= 0 && axes_batch_stride >= 9 && axes_row_stride >= 3, "gp_scalenet: bad sizes/strides");
    if (B == 0) return GP_OK;
    if (B <= num_sms()) return launch_scalenet<1>(p, axes, axes_batch_stride, axes_row_stride, pts_feat, B, length, as_stream(s));
    if (B < 8 * num_sms()) return launch_scalenet<2>(p, axes, axes_batch_stride, axes_row_stride, pts_feat, B, length, as_stream(s));
    return launch_scalenet<8>(p, axes, axes_batch_stride, axes_row_stride, pts_feat, B, length, as_stream(s));
}
