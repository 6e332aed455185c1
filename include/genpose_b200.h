/*
 * genpose_b200.h -- C ABI of libgenpose_b200.so: hand-written sm_100a CUDA kernels for the
 * per-object pose-generation hot path of GenPose++ (reference: PythonerJOJO/GenPose2).
 *
 * Conventions (SURVEY.md section 8(b)):
 *   - plain device pointers + sizes + an explicit cudaStream_t (passed as void*); no torch types;
 *   - the CALLER allocates every output and workspace (sizes from the gp_*_bytes() queries);
 *   - no hidden global state, re-entrant, the device is the one the pointers live on;
 *   - every entry returns 0 on success, a negative gp_status on bad arguments, or a positive
 *     cudaError_t if a launch failed.  Nothing ever calls exit() (the reference does:
 *     sampling_gpu.cu:248-252, ball_query_gpu.cu:62-65).  gp_last_error() gives the message.
 *   - all tensors are contiguous, float32 / int32 / float64 as stated per argument.
 *
 * Each entry cites the reference interface it replaces (paths relative to the reference root;
 * P2 = networks/pts_encoder/pointnet2_utils/pointnet2).
 */
#ifndef GENPOSE_B200_H
#define GENPOSE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void *gp_stream_t; /* cudaStream_t */

#if defined(__GNUC__)
#define GP_API __attribute__((visibility("default")))
#else
#define GP_API
#endif

enum gp_status {
    GP_OK = 0,
    GP_ERR_BAD_ARG = -1,
    GP_ERR_UNSUPPORTED = -2,
    GP_ERR_WORKSPACE = -3,
    GP_ERR_LAUNCH = -4
};

/* ABI version of this header (bumped on any signature change). */
GP_API int gp_version(void);
/* Message of the last failing call on this host thread (thread-local, never NULL). */
GP_API const char *gp_last_error(void);
/* Number of kernels launched by this library on this host thread since the last reset. */
GP_API long long gp_launch_count(void);
GP_API void gp_launch_count_reset(void);

/* ---------------------------------------------------------------------------------------------
 * (1) PointNet++ set-abstraction integer ops.  Indices are bit-exact with the reference ext.
 * ------------------------------------------------------------------------------------------ */

/* Replaces pointnet2_cuda.furthest_point_sampling_wrapper(b, n, m, points, temp, idx)
 * (P2/src/sampling.cpp:40-51 -> sampling_gpu.cu:93-253; Python: P2/pointnet2_utils.py:16-37).
 * xyz [B,N,3] f32 -> idx [B,m] i32.  No `temp` scratch: distances live in registers.
 * new_xyz (optional, may be NULL) [B,m,3] f32 receives xyz[b, idx[b,j], :] -- the fused
 * gather_operation of pointnet2_modules.py:43-47. */
GP_API int gp_fps(const float *xyz, int B, int N, int m, int32_t *idx, float *new_xyz, gp_stream_t s);
/* The same sampling for a cascade of levels (the encoder samples level k+1 from the centres of level k,
 * pointnet2_modules.py:43-47 called from pointnet2.py:115-121).  tie_free_out[b] = T: the first T - 1 sampling
 * steps of object b never had two different locations share the maximum distance.  tie_free_in (or NULL) must be
 * the tie_free_out of the call that produced `xyz` as its new_xyz: objects with tie_free_in[b] >= m get
 * idx = 0..m-1 (FPS of an FPS-ordered cloud is its own prefix when no step tied), the others are sampled. */
GP_API int gp_fps_chain(const float *xyz, int B, int N, int m, int32_t *idx, float *new_xyz,
                        const int32_t *tie_free_in, int32_t *tie_free_out, gp_stream_t s);

/* Replaces pointnet2_cuda.gather_points_wrapper(b, c, n, npoints, points, idx, out)
 * (P2/src/sampling.cpp:13-25 -> sampling_gpu.cu:8-43).  points [B,C,N], idx [B,m] -> out [B,C,m]. */
GP_API int gp_gather(const float *points, const int32_t *idx, int B, int C, int N, int m, float *out,
              gp_stream_t s);

/* Replaces pointnet2_cuda.ball_query_wrapper(b, n, m, radius, nsample, new_xyz, xyz, idx)
 * (P2/src/ball_query.cpp:16-27 -> ball_query_gpu.cu:9-66).  xyz [B,N,3], new_xyz [B,M,3] ->
 * idx [B,M,nsample] i32.  Every slot is written (the caller need not zero-initialise). */
GP_API int gp_ball_query(const float *new_xyz, const float *xyz, int B, int N, int M, float radius,
                  int nsample, int32_t *idx, gp_stream_t s);

/* Two radii in one scan of the cloud (the MSG grouper pair of pointnet2_modules.py:104-121). */
GP_API int gp_ball_query2(const float *new_xyz, const float *xyz, int B, int N, int M, float radius0,
                   int nsample0, int32_t *idx0, float radius1, int nsample1, int32_t *idx1,
                   gp_stream_t s);

/* gp_ball_query2 with the encoder's per-centre by-products written by the same launch (one thread owns one
 * centre): rel [B,M,3] = new_xyz - shift[b] (the centres in the object frame the hoisted first layers use,
 * replaces a torch subtraction) and tail [B,M,4] = [rel | 0] or, with tail_absolute, [new_xyz | 0] -- the last
 * four columns of the next level's channels-last rows [feat | xyz | 0] (replaces the torch.cat of
 * P2/pointnet2_utils.py:286-291).  shift [B,3] (NULL: zero), rel / tail may be NULL. */
GP_API int gp_ball_query2_tails(const float *new_xyz, const float *xyz, int B, int N, int M, float radius0,
                         int nsample0, int32_t *idx0, float radius1, int nsample1, int32_t *idx1,
                         const float *shift, float *rel, float *tail, int tail_absolute, gp_stream_t s);

/* Replaces pointnet2_cuda.group_points_wrapper(b, c, n, npoints, nsample, points, idx, out)
 * (P2/src/group_points.cpp:26-37 -> group_points_gpu.cu:47-89).
 * points [B,C,N], idx [B,M,nsample] -> out [B,C,M,nsample]. */
GP_API int gp_group(const float *points, const int32_t *idx, int B, int C, int N, int M, int nsample,
             float *out, gp_stream_t s);

/* Replaces QueryAndGroup.forward after the ball query (P2/pointnet2_utils.py:279-296): the two
 * grouping_operation calls, the xyz transpose, the recentring and the concat, in one pass.
 * xyz [B,N,3], new_xyz [B,M,3], features [B,C,N] (NULL when C == 0), idx [B,M,nsample] ->
 * out [B,3+C,M,nsample] with out[:, :3] = xyz[idx] - new_xyz and out[:, 3:] = features[idx]. */
GP_API int gp_query_group(const float *xyz, const float *new_xyz, const float *features,
                   const int32_t *idx, int B, int C, int N, int M, int nsample, float *out,
                   gp_stream_t s);

/* Channels-last ("one GEMM row per sample") form of the same QueryAndGroup tail, used by the drop-in
 * encoder so that the SharedMLP (conv1x1 + BN + ReLU, P2/pytorch_utils.py:5-33) is a plain row-major
 * GEMM chain.  feat_cl is [B,N,C] (channels last; NULL when C == 0), out is [B*M*nsample, ld_out] with
 * out[row, 0:3] = xyz[idx] - new_xyz, out[row, 3:3+C] = feat_cl[idx, :], zero padding up to ld_out. */
GP_API int gp_group_rows(const float *xyz, const float *new_xyz, const float *feat_cl, const int32_t *idx,
                  int B, int C, int N, int M, int nsample, int ld_out, float *out, gp_stream_t s);

/* Replaces F.max_pool2d(new_features, kernel_size=[1, nsample]) (P2/pointnet2_modules.py:59-61) on the
 * channels-last layout: h [G*nsample, C] -> out[g, 0:C] = max over the nsample rows of group g
 * (out has row stride ld_out so both MSG scales can land in one concatenated tensor). */
GP_API int gp_maxpool_rows(const float *h, long long G, int nsample, int C, int ld_out, float *out, gp_stream_t s);

/* A whole set-abstraction scale WITHOUT point features (the first level of Pointnet2ClsMSG(0)), fused:
 * grouping (xyz[idx] - new_xyz, P2/pointnet2_utils.py:279-282) -> SharedMLP 3 -> C1 -> C2 -> C3
 * (P2/pytorch_utils.py:5-33, BatchNorm folded by the caller: weights[i] is [Cout,Cin] row-major, biases[i]
 * [Cout]) -> max over nsample (P2/pointnet2_modules.py:59-61).  out[(b*M + p) * ld_out + c], c < C3.
 * FP32 FFMA (channels are too narrow for a tensor-core tile).  Instantiated specs: 16-16-32, 32-32-64;
 * nsample 16 or 32. */
GP_API int gp_sa_small_mlp(const float *xyz, const float *new_xyz, const int32_t *idx, int B, int N, int M,
                    int nsample, const float *const *weights, const float *const *biases, int C1, int C2, int C3,
                    float *out, int ld_out, gp_stream_t s);
/* The same scale with HOST copies of the folded weights: they travel in the launch's parameter space (constant
 * bank), so the kernel's FFMAs take them as constant operands instead of loading them from shared memory. */
GP_API int gp_sa_small_mlp_hostw(const float *xyz, const float *new_xyz, const int32_t *idx, int B, int N, int M,
                    int nsample, const float *const *host_weights, const float *const *host_biases, int C1, int C2,
                    int C3, float *out, int ld_out, gp_stream_t s);

/* gp_sa_small_mlp_hostw that also copies tail_src[(b*M + p), 0:4] ([x y z 0] of the centre) to
 * out[(b*M + p) * ld_out + tail_col .. + 3]: the level buffer [feat | xyz | 0] is complete after the launch. */
GP_API int gp_sa_small_mlp_hostw_tail(const float *xyz, const float *new_xyz, const int32_t *idx, int B, int N, int M,
                    int nsample, const float *const *host_weights, const float *const *host_biases, int C1, int C2,
                    int C3, float *out, int ld_out, const float *tail_src, int tail_col, gp_stream_t s);

/* Stream-ordered zero fill (a memset node, no kernel): the zero-initialisation the pooled GEMM outputs need. */
GP_API int gp_zero(void *dst, size_t bytes, gp_stream_t s);

/* One SharedMLP layer (P2/pytorch_utils.py:5-33: conv1x1 + BatchNorm(eval) folded + ReLU) on channels-last
 * rows, on the tcgen05 tensor cores: Y = relu(X . W^T + bias), optionally fused with the max-pool over
 * `pool_ns` consecutive rows (P2/pointnet2_modules.py:59-61).
 *   npass = 1: bf16 operands (bf16 mode);  npass = 3: fp32 values split into hi + lo bf16 and accumulated
 *   as hi*hi + lo*hi + hi*lo (16 mantissa bits per operand, fp32 accumulation) -- the fp32-mode path;
 *   npass = 2: tf32 operands (both rounded to nearest tf32, 11 significand bits; tcgen05 kind::tf32, fp32
 *   accumulation), packed to the same size as npass = 3.  Other values: GP_ERR_BAD_ARG (gp_gemm_packed_bytes
 *   returns 0).  The same npass values hold for gp_gemm_linear, gp_gemm_gather_bias_relu and gp_sa_mlp2_fused(_xyz).
 *   W [N,K] fp32 row-major is packed once per checkpoint with gp_gemm_pack (gp_gemm_packed_bytes bytes).
 *   X [R, ldx] fp32, ldx %% 4 == 0, columns K..ldx-1 must be finite (they meet zero weights).
 *   pool_ns == 0: Y [R, ldy] with ldy = round_up(N, 32); columns N..ldy-1 are written as zeros.
 *   pool_ns  > 0: pooled [R / pool_ns, ld_pooled] (zero-initialised by the caller) receives the max. */
GP_API size_t gp_gemm_packed_bytes(int N, int K, int npass);
GP_API int gp_gemm_pack(const float *W, int N, int K, int npass, void *packed, gp_stream_t s);
GP_API int gp_gemm_bias_relu(const float *X, long long R, int ldx, const void *packed, const float *bias, int N,
                      int K, int npass, float *Y, int ldy, int pool_ns, float *pooled, int ld_pooled,
                      gp_stream_t s);

/* Y = X . W^T (no bias, no activation), same engine and packing as gp_gemm_bias_relu.  Used to hoist the first
 * SharedMLP layer of a scale from the (centre, sample) rows to the points: the layer is linear before its
 * ReLU, so  W0 . [xyz[idx] - new_xyz ; feat[idx]]  =  (W0 . [xyz ; feat])[idx]  -  W0_xyz . new_xyz,
 * nsample x fewer multiply-adds and no gathered activation matrix in HBM. */
GP_API int gp_gemm_linear(const float *X, long long R, int ldx, const void *packed, int N, int K, int npass,
                   float *Y, int ldy, gp_stream_t s);

/* The per-centre term of a hoisted first layer:  Q[r][k] = sum_j new_xyz[r][j] * w0_xyz_t[j][k] - b0[k]  for k < c1,
 * zero for c1 <= k < ldq.  new_xyz [rows,3], w0_xyz_t [3,c1] = the xyz columns of the folded first-layer weight,
 * transposed. */
GP_API int gp_centre_term(const float *new_xyz, long long rows, const float *w0_xyz_t, const float *b0, int c1,
                   float *Q, int ldq, gp_stream_t s);
/* The same, and tail_dst[r * ld_tail + 0..3] = tail_src[r * 4 + 0..3]: the centres' [x y z 0] rows land in the
 * tail of this level's buffer in the same launch. */
GP_API int gp_centre_term_tail(const float *new_xyz, long long rows, const float *w0_xyz_t, const float *b0, int c1,
                        float *Q, int ldq, const float *tail_src, float *tail_dst, int ld_tail, gp_stream_t s);

/* Second SharedMLP layer with the hoisted first layer applied on the fly in the operand loader:
 *   A[r][k] = relu(P[(r / rows_per_batch) * n_src + gidx[r]][k] - Q[r / q_ns][k]),   Y = relu(A . W^T + bias)
 * P [batches * n_src, ldp] = per-point first-layer pre-activations (gp_gemm_linear), gidx [R] = ball-query
 * indices (row r = (batch, centre, sample)), Q [R / q_ns, ldq] = W0_xyz . new_xyz - b0 per centre.
 * Output / pooling arguments as gp_gemm_bias_relu. */
GP_API int gp_gemm_gather_bias_relu(const float *P, int n_src, int ldp, const int32_t *gidx, long long R,
                             int rows_per_batch, const float *Q, int ldq, int q_ns, const void *packed,
                             const float *bias, int N, int K, int npass, float *Y, int ldy, int pool_ns,
                             float *pooled, int ld_pooled, gp_stream_t s);

/* Layers 2 and 3 of a set-abstraction scale and its max-pool in one persistent kernel (P2/pointnet2_modules.py:
 * 45-66): the gather of gp_gemm_gather_bias_relu, H = relu(A . W1^T + b1) kept on the SM (TMEM -> shared
 * memory A operand), pooled[g] = max over the pool_ns rows of group g of relu(H . W2^T + b2).  The
 * (centre, sample) activation matrices never exist in HBM.
 *   packed1 = gp_gemm_pack(W1 [c2, c1]), packed2 = gp_gemm_pack(W2 [c3, c2]), same npass;
 *   c1 %% 4 == 0, c1 <= 256, c2 <= 384, c3 <= 512 (and within the shared-memory budget: fails loudly otherwise);
 *   pool_ns in {8, 16, 32}; pooled [R / pool_ns, ld_pooled], every element written once. */
GP_API int gp_sa_mlp2_fused(const float *P, int n_src, int ldp, const int32_t *gidx, long long R, int rows_per_batch,
                     const float *Q, int ldq, int q_ns, const void *packed1, const float *bias1, int c1, int c2,
                     const void *packed2, const float *bias2, int c3, int npass, int pool_ns, float *pooled,
                     int ld_pooled, gp_stream_t s);
/* The same kernel for a scale WITHOUT point features (the first level): the K = 3 first layer is evaluated in the
 * operand loader, A[r][k] = relu(W0[k] . (xyz[batch(r), gidx[r]] - centres[r / q_ns]) + b0[k]), one row per thread, so
 * neither the per-point table P nor Q exists.  xyz [batches, n_src, 3], centres [R / q_ns, 3] (new_xyz) on the device;
 * host_W0 [c1, 3] / host_b0 [c1] = HOST copies of the folded first layer (they travel in the launch's parameter space,
 * like gp_sa_small_mlp_hostw), c1 = 16 or 32; the rest as gp_sa_mlp2_fused. */
GP_API int gp_sa_mlp2_fused_xyz(const float *xyz, const float *centres, int n_src, const int32_t *gidx, long long R,
                         int rows_per_batch, int q_ns, const float *host_W0, const float *host_b0, const void *packed1,
                         const float *bias1, int c1, int c2, const void *packed2, const float *bias2, int c3, int npass,
                         int pool_ns, float *pooled, int ld_pooled, gp_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * (2)(3) ScoreNet / EnergyNet trunk.  Raw parameters in the reference's state-dict layout
 * (SURVEY.md section 5): nn.Linear weights are [out,in] row-major.
 * ------------------------------------------------------------------------------------------ */
typedef struct gp_trunk_params {
    const float *pose_w0;    /* pose_encoder.0.weight [256,9]    (scorenet.py:133-138) */
    const float *pose_b0;    /* pose_encoder.0.bias   [256] */
    const float *pose_w1;    /* pose_encoder.2.weight [256,256] */
    const float *pose_b1;    /* pose_encoder.2.bias   [256] */
    const float *fourier_w;  /* t_encoder.0.W         [64]       (scorenet.py:77-88) */
    const float *t_w;        /* t_encoder.1.weight    [128,128] */
    const float *t_b;        /* t_encoder.1.bias      [128] */
    const float *head_w0[3]; /* fusion_tail_{rot_x,rot_y,trans}.0.weight [256,1408] */
    const float *head_b0[3]; /* ....0.bias [256] */
    const float *head_w1[3]; /* ....2.weight [3,256] */
    const float *head_b1[3]; /* ....2.bias [3] */
} gp_trunk_params;

/* Bytes of the packed trunk (re-laid-out weights the kernels read; caller-allocated, device). */
GP_API size_t gp_trunk_packed_bytes(void);
/* Packs `raw` (device pointers) into `packed`.  Do once per checkpoint. */
GP_API int gp_trunk_pack(const gp_trunk_params *raw, void *packed, gp_stream_t s);
/* The blob of tf32 mode (mode 3 of the trunk entries): the same size and layout as gp_trunk_pack's, except that the
 * tensor-core weight images hold tf32 values (cvt.rna: round to nearest on the 13 dropped bits, ties away from zero)
 * with the two images of a 64-k chunk holding k 0..31 and k 32..63 instead of bf16 hi and lo parts.  The fp32
 * matrices, biases and output layers are identical, so gp_trunk_project accepts either blob.
 * Mode 3 needs a blob from gp_trunk_pack_tf32, modes 0..2 one from gp_trunk_pack.  The library cannot tell them
 * apart without reading device memory: passing the wrong kind is the caller's error and gives wrong results. */
GP_API int gp_trunk_pack_tf32(const gp_trunk_params *raw, void *packed, gp_stream_t s);

/* Per-object hoisted head projection: proj[b, 0:768] = head_w0[:, :1024] @ pts_feat[b] + head_b0
 * (the pts_feat columns of scorenet.py:249,259-261, constant over hypotheses and ODE stages).
 * pts_feat [B,1024] f32 -> proj [B,768] f32. */
GP_API int gp_trunk_project(const void *packed, const float *pts_feat, int B, float *proj, gp_stream_t s);

/* One PoseScoreNet.forward (scorenet.py:215-275): x [N,9] f32, t [N] f32 (one value per row),
 * proj [B,768] with row i belonging to object i / rows_per_object -> score [N,9] f32
 * (= f_theta / (std + 1e-7)).  Used by GFObjectPose.forward(mode="score") (posenet.py:305-307).
 * mode: 0 = fp32 FFMA, 1 = bf16 tcgen05, 2 = split-bf16 x3 tcgen05 (fp32-class), 3 = tf32 tcgen05, as for
 * gp_scorenet_ode. */
GP_API int gp_scorenet_eval(const void *packed, const float *proj, const float *x, const float *t, int N,
                     int rows_per_object, float *score, int mode, gp_stream_t s);

/* Flags that may be OR-ed into the `mode` argument of gp_scorenet_eval / _ode / _ode_dense / _pc / gp_energy when it
 * selects a tensor-core arithmetic (1, 2 or 3).  The tensor-core evaluator has two shapes: a 4-CTA cluster per 128-row
 * tile (shortest critical path; every CTA re-evaluates the pose encoder and integrates a private copy of the state)
 * and one CTA per tile (no redundant work, one state copy: the throughput shape).  Default: one CTA per tile when the
 * batch has more than 32 tiles (more than the GPU holds clusters at once), clusters otherwise. */
enum gp_mode_flag {
    GP_MODE_SOLO = 16,    /* force one CTA per tile */
    GP_MODE_CLUSTER = 32, /* force a 4-CTA cluster per tile */
    GP_MODE_SMEM_A = 64   /* one-CTA-per-tile shape: keep the activations (A operand) in shared memory instead of tensor memory
                             (modes 1 and 2 only: with mode 3 the entries return GP_ERR_UNSUPPORTED) */
};

/* Integrator statistics written by gp_scorenet_ode (device, 16 doubles). */
enum gp_ode_stat {
    GP_STAT_NFEV = 0,      /* RHS evaluations inside the solver (scipy res.nfev) */
    GP_STAT_ACCEPTED = 1,  /* accepted steps (res.t.size - 1) */
    GP_STAT_REJECTED = 2,
    GP_STAT_STATUS = 3,    /* 0 finished, -1 step size underflow, -2 attempt cap hit */
    GP_STAT_T_FINAL = 4,
    GP_STAT_H_INITIAL = 5,
    GP_STAT_H_LAST = 6,
    /* 8..24: cycle counters of the kernel's phases, CTA 0 (profiling aid, profiles/phase_breakdown.py) */
    GP_STAT_COUNT = 32
};

/* Bytes of device workspace gp_scorenet_ode needs for N rows. */
GP_API size_t gp_scorenet_ode_workspace_bytes(int N);

/* Replaces cond_ode_sampler (networks/gf_algorithms/samplers.py:180-258) including the host
 * scipy.integrate.solve_ivp(RK45) loop (samplers.py:226-234), the denoise step (:238-249),
 * Gram-Schmidt (:251-257) and `+ pts_center`: a device-resident Dormand-Prince 5(4) integrator
 * with scipy's step-size control shared over the flattened batch, fused with the ScoreNet RHS.
 *   x0          [N,9] f64   initial state  (= prior(T) [+ init_x], samplers.py:197-201)
 *   proj        [B,768] f32 from gp_trunk_project;   row i -> object i / rows_per_object
 *   pts_center  [N,3] f32
 *   T, eps, rtol, atol      as in the reference call (posenet.py:253-266)
 *   denoise     0/1
 *   x_out       [N,9] f64   final pose (normalised rotation, centre added); all NaN when the integration failed
 *                           (stats[GP_STAT_STATUS] != 0: step size underflow or attempt cap) -- the reference ignores
 *                           solve_ivp's status (samplers.py:226-236), this library poisons the result in band
 *   traj        NULL, or [max_traj, N, 9] f64: raw state after every accepted step, slot 0 = x0
 *   stats       [GP_STAT_COUNT] f64 (device)
 *   mode        arithmetic of the MLP contractions: 0 = fp32 FFMA on CUDA cores; 1 = bf16 operands on tcgen05;
 *               2 = tcgen05 with every operand split into two bf16 (hi*hi + lo*hi + hi*lo, fp32 accumulation in
 *               TMEM: 16 mantissa bits per operand, indistinguishable from fp32 on the reference's fixtures);
 *               3 = tf32 operands on tcgen05 (kind::tf32, 11 significand bits, fp32 accumulation; `packed` from
 *               gp_trunk_pack_tf32).
 *               Modes 1..3 run as 4-CTA clusters per 128-row tile (cooperative launch) or one CTA per tile (gp_mode_flag).
 * The sampler kernels (this entry, gp_scorenet_ode_dense, gp_scorenet_pc) are persistent grids with a spin grid barrier,
 * launched cooperatively so that every CTA is resident.  The one process-wide switch this library reads is the
 * environment variable GP_NONCOOPERATIVE_LAUNCH=1 (read once): it drops the cooperative attribute for profilers that
 * cannot replay cooperative cluster launches; with it set NOTHING else may share the GPU with such a launch (the grid
 * is sized for an otherwise idle device).  Leave it unset in production.
 */
GP_API int gp_scorenet_ode(const void *packed, const float *proj, const double *x0,
                    const float *pts_center, int N, int rows_per_object, double T, double eps,
                    double rtol, double atol, int denoise, double *x_out, double *traj,
                    int max_traj, double *stats, void *workspace, size_t workspace_bytes, int mode,
                    gp_stream_t s);

/* The same integration with scipy's dense output on a fixed grid (solve_ivp(..., t_eval=np.linspace(T, eps, num_steps)),
 * samplers.py:222-235; RkDenseOutput, scipy rk.py:715-737): every requested time is interpolated by the accepted step
 * that reaches it, y(te) = y_old + h * (K^T P) . [x, x^2, x^3, x^4], x = (te - t_old) / h.
 *   t_eval  [n_eval] f64 (device), in integration order (t_eval[0] = T, t_eval[n_eval-1] = eps)
 *   dense   [n_eval, N, 9] f64: raw states at t_eval (feed to gp_traj_finalize for the reference's `xs`)
 * The final pose is taken from the last interpolated state and the denoise step is (1 - eps) / n_eval, as
 * samplers.py:236-249 does when num_steps is given. */
GP_API int gp_scorenet_ode_dense(const void *packed, const float *proj, const double *x0,
                          const float *pts_center, int N, int rows_per_object, double T, double eps,
                          double rtol, double atol, int denoise, double *x_out, const double *t_eval,
                          int n_eval, double *dense, double *stats, void *workspace, size_t workspace_bytes,
                          int mode, gp_stream_t s);

/* Per-object step control.  The entries above share one step size and one RMS error norm over the whole flattened
 * batch (scipy's controller applied to all N*9 components), so an object's poses depend on which other objects share
 * the call.  These entries integrate every object as if the sampler had been called with that object alone: its own
 * select_initial_step, t, h, error norm over its R*9 components, accept / reject sequence, denoise step and
 * statistics.  Object b (rows b*R .. b*R+R-1, R = rows_per_object, N = B*R) is integrated start to end by one CTA (or
 * one 4-CTA cluster) on its own 128-row tile; the result is bit-identical to a gp_scorenet_ode call with that object
 * alone on the same evaluator shape.  The tensor-core shape follows the tile count B by the batch rule (clusters for
 * B <= 32, one CTA per object above); GP_MODE_SOLO / GP_MODE_CLUSTER force it.
 *   rows_per_object  R <= 128 (GP_ERR_UNSUPPORTED above: an object spanning tiles is not supported)
 *   stats       [GP_STAT_COUNT] f64 (device): summary -- nfev is the maximum over objects, accepted / rejected are
 *               sums, status is the first non-zero one; t_final / h_initial / h_last are those of that object
 *               (object 0 when none failed)
 *   obj_stats   [B, GP_STAT_COUNT] f64 (device): the statistics of each object, fields as in gp_ode_stat
 *   x_out       [N,9] f64; the rows of a failed object (status != 0) are NaN, the other objects are unaffected
 * The trajectory of accepted steps is not offered (objects accept different numbers of steps); the dense-output
 * variant takes a grid common to all objects.  The other arguments are those of gp_scorenet_ode / _dense. */
GP_API size_t gp_scorenet_ode_objects_workspace_bytes(int B, int R);
GP_API int gp_scorenet_ode_objects(const void *packed, const float *proj, const double *x0,
                            const float *pts_center, int N, int rows_per_object, double T, double eps,
                            double rtol, double atol, int denoise, double *x_out, double *stats, double *obj_stats,
                            void *workspace, size_t workspace_bytes, int mode, gp_stream_t s);
GP_API int gp_scorenet_ode_dense_objects(const void *packed, const float *proj, const double *x0,
                                  const float *pts_center, int N, int rows_per_object, double T, double eps,
                                  double rtol, double atol, int denoise, double *x_out, const double *t_eval,
                                  int n_eval, double *dense, double *stats, double *obj_stats, void *workspace,
                                  size_t workspace_bytes, int mode, gp_stream_t s);
/* Per-object start time: the arguments of gp_scorenet_ode_dense_objects, except that
 *   T_obj   [B] f64 (device) replaces T: object b is integrated from T_obj[b] to eps.  The caller must ensure
 *           T_obj[b] > eps (this entry cannot read device memory); NULL is rejected.
 *   t_eval  optional, per object: [B, n_eval] f64 (device), row b in integration order (t_eval[b][0] = T_obj[b]);
 *           NULL (with dense NULL) means no dense output.  dense is [n_eval, N, 9] as in the entries above.
 * The denoise step is (1 - eps) / n_eval with dense output, (1 - eps) / 1000 without.  Workspace:
 * gp_scorenet_ode_objects_workspace_bytes(B, R).  The entries above are this one with T_obj[b] = T for every object
 * (bit for bit). */
GP_API int gp_scorenet_ode_objects_t0(const void *packed, const float *proj, const double *x0,
                               const float *pts_center, int N, int rows_per_object, const double *T_obj, double eps,
                               double rtol, double atol, int denoise, double *x_out, const double *t_eval,
                               int n_eval, double *dense, double *stats, double *obj_stats, void *workspace,
                               size_t workspace_bytes, int mode, gp_stream_t s);

/* Keyed per-object initial noise of the ODE sampler (DESIGN.md section 4.6f): noise [B*R, 9] f32 (device), where the
 * block of object b (rows b*R .. b*R+R-1) depends only on keys[b] and sigma[b], never on b, B or the other keys.
 *   keys    [B] int64 (device);  sigma [B] f32 (device): the standard deviation of object b's block.
 * Definition: Philox4x32-10 keyed with (lo32, hi32) of keys[b].  Element e = r*9 + c of the block belongs to Box-Muller
 * pair p = e / 2; pair p uses the words 2*(p % 2) and 2*(p % 2) + 1 of the Philox output for counter (p / 2, 0, 0, 0).
 * The words give u_a, u_b = (w + 0.5) * 2^-32 (f64); n_2p = sqrt(-2 ln u_a) cos(2 pi u_b) and n_2p+1 = sqrt(-2 ln u_a)
 * sin(2 pi u_b) in f64, rounded to f32.  The output is n * sigma[b], multiplied in f32 (as ve_prior scales its f32
 * normals).  R*9 odd: the sine of the last pair is dropped. */
GP_API int gp_object_noise(const int64_t *keys, const float *sigma, int B, int R, float *noise, gp_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * Per-object point clouds from a depth frame and an instance-label image (DESIGN.md section 4.13): the `pts` /
 * `pts_center` inputs the pipeline takes, built on the device instead of the datasets' numpy loop
 * (datasets/datasets_omni6dpose.py:459-473).
 * ------------------------------------------------------------------------------------------ */

/* Most objects and pixels one gp_backproject_instances or gp_backproject_frames call takes (2^30 pixels keeps every
 * pixel index of the 1024-pixel tiles inside int), and most frames one gp_backproject_frames call takes. */
enum { GP_MAX_FRAME_OBJECTS = 1024, GP_MAX_FRAME_PIXELS = 1 << 30, GP_MAX_FRAMES = 1024 };

/* Stage A, back-projection and stable per-object compaction.
 *   depth  [H,W] f32 metres;  labels [H,W] i32: value b+1 is object b, values outside 1..B are background.
 *   Pixel (u = column, v = row) is kept iff its label is in 1..B and z = depth > 0 and finite; its point is
 *   (x, y, z) with x = ((float)u - cx) * z / fx and y = ((float)v - cy) * z / fy, IEEE float32 in that order
 *   (no pixel-centre offset).
 *   xyz     [H*W, 3] f32 (capacity-sized): object b's points are rows offsets[b] .. offsets[b+1]-1 in row-major
 *           pixel order (numpy's xyz[labels == b+1]); rows from offsets[B] on are not written.
 *   offsets [B+1] i32 (device).
 * B > GP_MAX_FRAME_OBJECTS returns GP_ERR_UNSUPPORTED, H * W > GP_MAX_FRAME_PIXELS GP_ERR_BAD_ARG (the workspace
 * query returns 0 for both, as for bad sizes).  Intrinsics
 * must be finite with fx, fy != 0.  Three kernel launches, no host synchronisation. */
GP_API size_t gp_backproject_instances_workspace_bytes(int H, int W, int B);
GP_API int gp_backproject_instances(const float *depth, const int32_t *labels, int H, int W, float fx, float fy,
                                    float cx, float cy, int B, float *xyz, int32_t *offsets, void *workspace,
                                    size_t workspace_bytes, gp_stream_t s);

/* Stage A over F frames of one size in one pass (a batch of tracked videos, a multi-camera rig).
 *   depth [F,H,W] f32, labels [F,H,W] i32, intrinsics [F][4] f32 (fx, fy, cx, cy of each frame, device),
 *   frame_offsets [F+1] i32 (device): frame f holds the objects frame_offsets[f] .. frame_offsets[f+1]-1, numbered
 *   frame-major; label l of frame f with 1 <= l <= n_f = frame_offsets[f+1] - frame_offsets[f] is object
 *   frame_offsets[f] + l - 1, any other label (one above n_f too) is background.  Pixel rules and arithmetic are
 *   gp_backproject_instances', with the pixel's own frame's intrinsics.
 *   xyz [F*H*W, 3] f32 (capacity-sized), offsets [B+1] i32: bit for bit the concatenation, in frame order, of F
 *   gp_backproject_instances calls (object b in rows offsets[b] .. offsets[b+1]-1, row-major pixel order of its frame).
 * frame_offsets is never read on the host, so one captured graph replays new per-frame object counts.  Whatever it
 * holds, the kernels read and write in bounds: frame_offsets[0] is taken as 0 and frame_offsets[F] as B, and each
 * frame_offsets[f] in between is raised to the largest of frame_offsets[1..f] and clamped into [0, B] (malformed
 * offsets give wrong clouds, never an out-of-bounds access).  Zero or non-finite intrinsics give non-finite points.
 * B > GP_MAX_FRAME_OBJECTS or F > GP_MAX_FRAMES returns GP_ERR_UNSUPPORTED, F * H * W > GP_MAX_FRAME_PIXELS
 * GP_ERR_BAD_ARG (the workspace query returns 0 for these and for bad sizes).  Workspace:
 * (B * ceil(H*W / 1024) + B + F + 1) ints.  Three kernel launches, no host synchronisation; with F = 1, objects
 * [0, B) and the same intrinsics the result equals gp_backproject_instances'. */
GP_API size_t gp_backproject_frames_workspace_bytes(int F, int H, int W, int B);
GP_API int gp_backproject_frames(const float *depth, const int32_t *labels, int F, int H, int W,
                                 const float *intrinsics, const int32_t *frame_offsets, int B, float *xyz,
                                 int32_t *offsets, void *workspace, size_t workspace_bytes, gp_stream_t s);

/* Stage B, sample_points (datasets_omni6dpose.py:459-473) with a keyed random choice.  Object b has the K points
 * xyz[offsets[b] .. offsets[b+1]-1] (offsets clamped into [0, rows] first; K = 0 when they cross); pts [B,N,3] f32:
 *   K < N: row r < (N / K) * K is point r % K (np.tile), the last N % K rows are points pi_b(0) .. pi_b(N % K - 1);
 *   K == N: the cloud unchanged;  K > N: row j is point pi_b(j) (permutation(K)[:N]);
 *   K == 0: zero rows and a zero centre.
 * pi_b, a permutation of [0, K): a 4-round balanced Feistel network on k = max(2, ceil(log2 K)) bits, k rounded up
 * to even, halves of k/2 bits (x = L << k/2 | R); round r = 0..3 maps (L, R) to (R, L ^ F_r(R)) with
 * F_r(R) = Philox4x32-10(counter (R, r, 1, 0), key (lo32, hi32) of keys[b]).x & (2^(k/2) - 1); values >= K are
 * encrypted again (cycle walking).  Counter word 2 = 1 keeps this stream apart from gp_object_noise's (q, 0, 0, 0).
 *   pts_center [B,3] f32: the mean of the N rows, summed in float64 and rounded to float32 (within 1 float32 ulp of
 *   the float64 mean of pts);  counts [B] i32: K.
 *   keys [B] int64 (device).  xyz may be NULL when rows == 0. */
GP_API int gp_sample_points(const float *xyz, long long rows, const int32_t *offsets, const int64_t *keys, int B,
                            int N, float *pts, float *pts_center, int32_t *counts, gp_stream_t s);

/* Post-processing of a recorded trajectory into the reference's `xs` (samplers.py:251-255):
 * traj [S,N,9] f64 raw -> xs [N,S,9] f64 with Gram-Schmidt on the rotation part and the centre
 * added. */
GP_API int gp_traj_finalize(const double *traj, const float *pts_center, int S, int N, double *xs,
                     gp_stream_t s);

/* Replaces cond_pc_sampler (samplers.py:113-177): num_steps x {Langevin corrector, Euler-Maruyama
 * predictor}, time grid linspace(1, eps, num_steps), one batch-wide step-size reduction per step.
 *   x0 [N,9] f32; noise [num_steps,2,N,9] f32 (the torch.randn_like draws in call order);
 *   time_steps [num_steps] f32 (device) = torch.linspace(1.0, eps, num_steps) (samplers.py:129);
 *   xs NULL or [N,num_steps,9] f32; mean_x [N,9] f32. */
GP_API size_t gp_scorenet_pc_workspace_bytes(int N);
GP_API int gp_scorenet_pc(const void *packed, const float *proj, const float *x0, const float *noise,
                   const float *pts_center, const float *time_steps, int N, int rows_per_object,
                   int num_steps, double snr, float *xs, float *mean_x, void *workspace,
                   size_t workspace_bytes, int mode, gp_stream_t s);

/* Replaces PoseNet.get_energy's network call + PoseEnergyNet.get_energy
 * (posenet_agent.py:660-705, energynet.py:151-208; energy_mode=IP, s_theta_mode=score,
 * norm_energy=identical).  poses [N,9] f64 camera frame; the centre is subtracted from the
 * translation (posenet_agent.py:694), the pose cast to f32 (:668-670).  t_rows [N] f32.
 * -> energy [N,2] f32 = [E_rot, E_trans]. */
GP_API int gp_energy(const void *packed, const float *proj, const double *poses, const float *pts_center,
              const float *t_rows, int N, int rows_per_object, float *energy, int mode, gp_stream_t s);

/* ---------------------------------------------------------------------------------------------
 * (4) Energy-ranked outlier rejection + quaternion averaging + DBSCAN, and the ScaleNet head.
 * ------------------------------------------------------------------------------------------ */

/* Replaces sort_poses_by_energy (networks/reward.py:131-155) + the aggregation block
 * (runners/evaluation_single.py:179-215 = evaluation_tracking.py:146-183 = infer.py:158-194):
 * rot / trans ranked independently by their energy channel, top `retain` kept, 6D -> quaternion,
 * eigen-average (utils/misc.py:295-317), DBSCAN(eps, min_samples) on the rows of the
 * 1 - <qi,qj>^2 matrix, largest cluster re-averaged, mean translation.
 *   poses [B,R,9] f64, energy [B,R,2] f32 -> pose_out [B,4,4] f32;
 *   labels_out NULL or [B,retain] i32 (DBSCAN labels, for inspection);
 *   sorted_out NULL or [B,R,9] f64 (sort_poses_by_energy's first return value).
 * Requires R <= 64 and retain <= 32 (retain <= 64 when clustering == 0: plain quaternion average + mean
 * translation over all hypotheses, posenet_agent.py:561-570 return_average_res). */
GP_API int gp_aggregate(const double *poses, const float *energy, int B, int R, int retain,
                 int clustering, double clustering_eps, int min_samples, float *pose_out,
                 int32_t *labels_out, double *sorted_out, gp_stream_t s);

/* Replaces the tail of PoseNet.pred_func (networks/posenet_agent.py:547-559): get_rot_matrix (utils/misc.py:121-160:
 * rotation_6d_to_matrix(.).permute(0,2,1)) + matrix_to_quaternion (utils/transforms/rotation_conversions.py:102-161)
 * + cat with the translation.  poses [N,9] f64 -> out [N,7] f64 = [q_wxyz | t]. */
GP_API int gp_pose_to_quat(const double *poses, int N, double *out, gp_stream_t s);

typedef struct gp_scalenet_params {
    const float *axes_w0; /* axes_encoder.0.weight [256,180] (networks/scalenet.py:20-25) */
    const float *axes_b0;
    const float *axes_w1; /* axes_encoder.2.weight [256,256] */
    const float *axes_b1;
    const float *tail_w0; /* fusion_tail_length.0.weight [256,1280] */
    const float *tail_b0;
    const float *tail_w1; /* fusion_tail_length.2.weight [3,256] */
    const float *tail_b1;
} gp_scalenet_params;

/* Replaces ScaleNet.forward (networks/scalenet.py:33-49) + encode_axes
 * (utils/genpose_utils.py:8-18).  axes [B,3,3] f32 (row stride `axes_stride` floats, so the
 * [:3,:3] block of a [B,4,4] pose can be passed with stride 4 and batch stride 16),
 * pts_feat [B,1024] -> length [B,3]. */
GP_API int gp_scalenet(const gp_scalenet_params *p, const float *axes, int axes_batch_stride,
                int axes_row_stride, const float *pts_feat, int B, float *length, gp_stream_t s);

#ifdef __cplusplus
}
#endif
#endif /* GENPOSE_B200_H */
