/* libserl_b200 - C ABI of the B200-native DrQ/SAC learner hot path.
 *
 * The reference (rail-berkeley/serl) has no FFI: its boundary is the Python API of `serl_launcher`
 * (SURVEY.md §8b).  This header is the C-ABI underneath this repo's Python mirror of that API
 * (serl_b200/): plain pointers and sizes, an explicit CUDA stream (cudaStream_t passed as void*),
 * no torch types, no allocation inside the library (callers own all buffers / workspaces).
 * Every function returns 0 on success or a negative SERL_ERR_* code; serl_last_error() gives the
 * message for the calling thread.  All pointers are DEVICE pointers unless a name says `host`.
 *
 * Citations are relative to /root/reference/serl_launcher/serl_launcher.
 */
#ifndef SERL_B200_H_
#define SERL_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SERL_MAX_CAMS 4

/* ---- library ------------------------------------------------------------------------------- */
const char* serl_last_error(void);
int serl_set_pdl(int enabled);                /* programmatic dependent launch for every kernel of the library (default: SERL_PDL env) */
int serl_stem_v2_active(void);                /* 1: the fused stem uses the TMA-im2col kernel (SERL_STEM_V2=1 and tensor map accepted) */
int serl_version(void);                       /* ABI version, bumped on signature changes */
unsigned long long serl_launch_count(void);   /* kernels this library has enqueued in this process (graph capture included) */
int serl_device_sm_count(int device);         /* host query used to size persistent grids */
int serl_balanced_grid(int items, int sms);   /* CTAs of a persistent one-CTA-per-SM kernel over `items` work items: the smallest grid with as few waves as min(items, sms) CTAs */

/* ---- replay ring in HBM ---------------------------------------------------------------------
 * Storage layout of data/replay_buffer.py:41-66 + data/memory_efficient_replay_buffer.py:13-51:
 * ONE camera frame per slot (frame dedup), per-slot scalars, a validity byte per slot. */
typedef struct serl_replay_view {
  const uint8_t* frames[SERL_MAX_CAMS];  /* (capacity, H, W, C) uint8 per camera                   */
  const float* state;                    /* (capacity, T*S) observations.state                      */
  const float* next_state;               /* (capacity, T*S) next_observations.state                 */
  const float* actions;                  /* (capacity, A)                                           */
  const float* rewards;                  /* (capacity,)                                             */
  const float* masks;                    /* (capacity,)                                             */
  const uint8_t* dones;                  /* (capacity,)                                             */
  const uint8_t* valid;                  /* (capacity,) _is_correct_index                           */
  int32_t num_cams, height, width, channels, num_stack /*T*/, state_dim /*S*/, action_dim /*A*/;
  int32_t capacity, size;                /* size = len(buffer): draws are uniform over [0, size)    */
} serl_replay_view;

typedef struct serl_sample_request {
  uint64_t seed, step;           /* Philox key / counter words of the index draw (repo spec)         */
  const uint64_t* step_dev;      /* optional device counter overriding `step` (CUDA-graph replay)     */
  const int32_t* size_dev;       /* optional device fill level overriding rv->size                    */
  uint32_t lane_offset;          /* Philox lane of output row 0                                      */
  int32_t batch;                 /* rows drawn by this call                                          */
  const int32_t* explicit_idx;   /* optional (batch): gather these slots instead of drawing          */
  const uint32_t* key_obs;       /* device uint32[2]: JAX key; frame g uses split(key, crop_total)[g] */
  const uint32_t* key_next;
  const int32_t* explicit_off_obs;   /* optional (crop_total, 2) [cy, cx] overriding the keys        */
  const int32_t* explicit_off_next;
  int32_t crop_total;            /* frames in the whole (possibly concatenated) batch = B_total * T   */
  int32_t out_row_offset;        /* first output row written by this call (RLPD: demo half offset)    */
  int32_t padding;               /* DrQ pad (4): offsets in [0, 2*padding]                            */
} serl_sample_request;

typedef struct serl_batch_out {
  uint8_t* obs_pix[SERL_MAX_CAMS];   /* (B_total, T, H, W, C) shifted observation frames             */
  uint8_t* next_pix[SERL_MAX_CAMS];  /* (B_total, T, H, W, C) shifted next-observation frames         */
  float* obs_state; float* next_state;   /* (B_total, T*S)                                           */
  float* actions; float* rewards; float* masks; uint8_t* dones;
  int32_t* idx;                      /* optional (B_total) drawn slots                                */
  int32_t* off_obs; int32_t* off_next;   /* optional (B_total*T, 2) applied offsets                   */
  int32_t* status;                   /* device int32, OR-ed with 1 if a draw found no valid slot      */
} serl_batch_out;

/* Replaces MemoryEfficientReplayBuffer.sample (memory_efficient_replay_buffer.py:91-164) +
 * ReplayBuffer.get_iterator's device_put (replay_buffer.py:77-90) + _unpack (utils/train_utils.py:44-66)
 * + batched_random_crop (vision/data_augmentations.py:7-36, agents/continuous/drq.py:244-253).
 * One-sided output: when every obs_pix[c] (or every next_pix[c]) is NULL only the other view's frames are gathered and
 * cropped (one CTA per row and camera instead of two); only that view's crop key / explicit offsets are needed.  The
 * reward classifier's batch (examples/async_cable_route_drq/train_reward_classifier.py) takes positive rows' next frames and negative rows' frames. */
int serl_replay_sample_crop(const serl_replay_view* rv, const serl_sample_request* rq,
                            const serl_batch_out* out, void* stream);

typedef struct serl_scatter_request {
  int32_t n;                         /* slot writes, applied independently (no ordering inside a call) */
  const int32_t* dst_slot;           /* (n)                                                            */
  const int32_t* src_slot;           /* (n)  >= 0: copy from that ring slot; < 0: from staging row k    */
  const uint8_t* frames[SERL_MAX_CAMS];  /* staging (n, H, W, C)                                       */
  const float* state; const float* next_state; const float* actions;
  const float* rewards; const float* masks; const uint8_t* dones;
  const uint8_t* valid;              /* (n) validity byte to store                                     */
  int64_t row_stride;                /* 0: the fields above are packed (n, ...) arrays; else they point into row 0 of an
                                      * interleaved staging record and row k lies k*row_stride BYTES further (the whole
                                      * staged batch then moves host->device as ONE copy)                          */
} serl_scatter_request;

/* Device side of MemoryEfficientReplayBuffer.insert (memory_efficient_replay_buffer.py:53-89,
 * replay_buffer.py:71-75): applies slot writes staged by the host ring logic. */
int serl_replay_scatter(const serl_replay_view* rv, const serl_scatter_request* rq, void* stream);
int serl_counter_add(uint64_t* counter, uint64_t inc, void* stream);   /* device-resident step counters */
int serl_replay_set_valid(uint8_t* valid, const int32_t* slots, const uint8_t* vals, int n, void* stream);
/* same + publishes the ring's new size to its device-resident copy (read by graph-replayed sampling launches) */
int serl_replay_commit(uint8_t* valid, const int32_t* slots, const uint8_t* vals, int n, int32_t* size_dev, int32_t size, void* stream);

/* ---- JAX-compatible key schedule and random fills ---------------------------------------------
 * Key slots written by serl_rng_schedule (uint32[2] each), following SACAgent.update's split order
 * (agents/continuous/sac.py:137,152,197,224,288; common/common.py:198-200; drq.py:307-308). */
enum {
  SERL_KEY_CROP_OBS = 0, SERL_KEY_CROP_NEXT = 1, SERL_KEY_CRITIC_NEXT = 2, SERL_KEY_CRITIC_SUBSAMPLE = 3,
  SERL_KEY_ACTOR_DROPOUT = 4, SERL_KEY_ACTOR_SAMPLE = 5, SERL_KEY_TEMP_NEXT = 6, SERL_NUM_KEYS = 8
};
int serl_rng_schedule(uint32_t* rng_state, uint32_t* keys, int do_aug, int do_update, void* stream);
int serl_normal_fill(const uint32_t* key, float* out, int n, void* stream);            /* jax.random.normal   */
int serl_dropout_mask_fill(const uint32_t* key, uint32_t fold, float keep, uint8_t* mask, int n, void* stream);
int serl_subsample_idx(const uint32_t* key, int ensemble, int32_t* out /*n*/, int n, void* stream); /* randint(key,(n,),0,E), sac.py:153-158 */

/* Host mirrors of the integer RNG specs (same code compiled for the host; usable without a GPU). */
int serl_host_rng_schedule(uint32_t* rng_state_host, uint32_t* keys_host, int do_aug, int do_update);
int serl_host_crop_offsets(const uint32_t key_host[2], int n_frames, int padding, int32_t* out_host);
int serl_host_draw_indices(uint64_t seed, uint64_t step, uint32_t lane_offset, int batch, int size,
                           const uint8_t* valid_host, int32_t* out_host);
int serl_host_threefry_split(const uint32_t key_host[2], int n, uint32_t* out_host);
int serl_host_random_bits(const uint32_t key_host[2], int size, uint32_t* out_host);

/* ---- frozen ResNet-10 trunk, fp32 build (vision/resnet_v1.py:217-286,129-156) ------------------ */
/* NHWC conv, HWIO weights, explicit low/high zero padding.  x_is_u8: x is uint8 and the ImageNet
 * normalisation (x/255 - mean)/std of resnet_v1.py:222-224 is fused into the operand load. */
int serl_conv2d_nhwc_f32(const void* x, int x_is_u8, const float* w, float* y, int N, int Hi, int Wi, int Ci,
                         int Co, int kh, int kw, int stride, int pad_lo, int pad_hi, void* stream);
/* GroupNorm (flax statistics), optional residual add and ReLU; y may alias x. */
int serl_groupnorm_nhwc_f32(const float* x, float* y, const float* scale, const float* bias, const float* residual,
                            int N, int HW, int C, int groups, float eps, int relu, void* stream);
int serl_maxpool3x3s2_nhwc_f32(const float* x, float* y, int N, int Hi, int Wi, int C, void* stream);

/* ---- frozen ResNet-10 trunk, 16-bit build on tcgen05 tensor cores (same layers as above) ---------- */
/* operand format of the kind::f16 MMAs: bf16, or fp16 (same throughput, 3 more mantissa bits; packs saturate) */
enum { SERL_FMT_BF16 = 0, SERL_FMT_FP16 = 1 };
/* uint8 crops (N,H,W,3) -> normalised 16-bit, 2x2 space-to-depth, zero padded: xs (N, H/2+3, W/2+3, 16)
 * (12 real channels (p,q,c) + 4 zero channels, so four taps are one aligned 128-byte operand row) */
int serl_trunk_stem_prep_h16(const uint8_t* x, void* xs, int N, int H, int W, int fmt, void* stream);
typedef struct serl_conv_tc_desc {
  const void* x;           /* 16-bit NHWC (N,Hi,Wi,Ci); stem: the space-to-depth image (Hi,Wi = its dims, Ci ignored) */
  const void* w;           /* 16-bit [Co][K], K-major, K = kh*kw*Ci (stem: 4 x 64 with 48 valid per row)             */
  void* y;                 /* 16-bit (N,Ho,Wo,Co) raw convolution output (pre-GroupNorm)                              */
  float* stats;            /* (N,4,2) fp32 sum / sum-of-squares per GroupNorm group, accumulated (pre-zero it)       */
  const float* in_a;       /* optional (N,Ci): operand transform relu(in_a*x + in_b) = previous GroupNorm + ReLU      */
  const float* in_b;
  int32_t* error;          /* device int32, OR-ed with 2 if a pipeline barrier timed out                             */
  int32_t N, Hi, Wi, Ci, Ho, Wo, Co, kh, kw, stride, pad_lo, stem, fmt;
} serl_conv_tc_desc;
int serl_conv2d_tc_h16(const serl_conv_tc_desc* d, void* stream);
/* Stride-1 3x3 SAME convolution without im2col redundancy: the input patch of a 128-position raster tile is staged once
 * in shared memory and the nine taps are shifted UMMA descriptors over it; weights arrive by TMA.  Same descriptor as
 * above (kh=kw=3, stride=1, pad_lo=1, no operand transform).  base_offset_mode: 0 = descriptor base_offset field left 0. */
int serl_conv3x3s1_tc_h16(const serl_conv_tc_desc* d, int base_offset_mode, void* stream);
/* conv_init (7x7/2 as a 4x4/1 conv over the space-to-depth image) FUSED with the 3x3/2 SAME max-pool that follows its
 * GroupNorm + ReLU (vision/resnet_v1.py:247-261).  relu(a*x+b) is monotone in x with the sign of the frozen GroupNorm
 * scale, so the pool runs on the raw sign-adjusted conv output inside the epilogue and the 64x64 map never reaches HBM.
 * xs (N,67,67,16) from serl_trunk_stem_prep_h16; w = packed stem weights; pooled (N,32,32,64); side (N,4,32,64);
 * stats (N,4,2) GroupNorm sums of the raw conv output; neg_mask bit c = (scale[c] < 0).
 * serl_pool_finish_h16 then writes y = relu(|a| * pooled' + b) with (a, b) from serl_gn_finalize. */
typedef struct serl_stem_pool_desc {
  const void* xs; const void* w; void* pooled; void* side; float* stats; int32_t* error;
  uint64_t neg_mask;
  int32_t N, fmt;
} serl_stem_pool_desc;
int serl_stem_conv_pool_tc_h16(const serl_stem_pool_desc* d, void* stream);
int serl_pool_finish_h16(const void* pooled, const void* side, const float* a, const float* b, void* y, int N, int fmt, void* stream);
/* "_gn" consumers: take the conv epilogue's GroupNorm sums (N,4,2) + the frozen scale / bias instead of a finalized (a, b)
 * table and derive the affine in registers (same arithmetic as serl_gn_finalize) - no finalize launch in the chain. */
int serl_pool_finish_gn_h16(const void* pooled, const void* side, const float* stats, const float* gamma, const float* beta, void* y,
                            int N, float eps, int fmt, void* stream);
int serl_affine_relu_gn_h16(void* x, const float* stats, const float* gamma, const float* beta, int N, int HW, int C, float eps, int fmt,
                            void* stream);
int serl_block_combine_gn_h16(const void* y2, const float* stats2, const float* gamma2, const float* beta2, const void* res,
                              const float* stats_r, const float* gamma_r, const float* beta_r, void* out_h16, float* out_f32,
                              int N, int HW, int C, float eps, int fmt, void* stream);
/* (N,4,2) sums -> per-(image, channel) affine a = rstd*gamma, b = beta - mean*a (flax GroupNorm statistics) */
int serl_gn_finalize(const float* stats, const float* gamma, const float* beta, float* out_a, float* out_b, int N, int C,
                     int HW, float eps, void* stream);
/* in place: x <- relu(a*x + b) (GroupNorm + ReLU of a raw conv output, materialised for the next conv's operand gather) */
int serl_affine_relu_h16(void* x, const float* a, const float* b, int N, int HW, int C, int fmt, void* stream);
int serl_maxpool_affine_h16(const void* x, const float* a, const float* b, void* y, int N, int Hi, int Wi, int C, int fmt, void* stream);
/* relu((a2*y2+b2) + residual), residual = res or ar*res+br; writes 16-bit (next block) or fp32 (final features) */
int serl_block_combine_h16(const void* y2, const float* a2, const float* b2, const void* res, const float* ar, const float* br,
                           void* out_h16, float* out_f32, int N, int HW, int C, int fmt, void* stream);

/* ---- dense algebra for the trainable heads (fp32) ---------------------------------------------- */
typedef struct serl_gemm_desc {
  const float* A; const float* B; float* C; const float* bias;
  float* workspace; size_t workspace_bytes;     /* split-K / batch-reduce partials */
  int32_t M, N, K, Z;
  int64_t sAz, sAm, sAk, sBz, sBk, sBn, sCz, sBiasZ;
  int32_t ldc;
  int32_t accumulate;                           /* C += result                                     */
  int32_t reduce_z;                             /* single C = sum over z                           */
} serl_gemm_desc;
int serl_gemm_f32(const serl_gemm_desc* d, void* stream);
/* Same contract on the tensor cores: fp32 operands split into TF32 hi + lo parts, three tcgen05.mma (kind::tf32) products
 * per k-step accumulated in fp32 TMEM ("3xTF32": fp32-class accuracy, ~2^-22 per product).  Heads of the 16-bit builds. */
int serl_gemm_tf32x3(const serl_gemm_desc* d, void* stream);

/* Heads of the 16-bit builds, round 2: single-pass TF32 GEMM (tcgen05 kind::tf32, operands by TMA straight from the fp32
 * tensors: X @ W, dZ @ W^T and X^T @ dZ of a Dense layer all read the row-major arrays in place) with fused epilogues.
 * Replaces, per launch, Dense (+ bias) [+ LayerNorm + tanh [+ value head | + policy heads + tanh-Gaussian sample]] of
 * networks/mlp.py:22-31, networks/actor_critic_nets.py:57-73,178-227,230-272, vision/resnet_v1.py:371-374.
 * C[z](m, n) = sum_k A[z](m, k) B[z](k, n); element strides in floats; per operand one of its two strides must be 1 and the
 * other a multiple of 4, base pointers 16-byte aligned (TMA), z stride 0 = the operand is shared by the Z members.
 * Up to SERL_TGEMM_MAX_PROBLEMS problems (same M, N, K, operand layouts and epilogue) per launch. */
#define SERL_TGEMM_MAX_PROBLEMS 6
#define SERL_TGEMM_EPI_STORE 0            /* C = acc + bias (+ C)                                                        */
#define SERL_TGEMM_EPI_LN_TANH 1          /* N == 256: C = tanh(LayerNorm(acc + bias) * scale + ln_bias); optional xhat, rstd */
#define SERL_TGEMM_EPI_LN_TANH_HEAD 2     /* ... and head_out[m, :head_n] = C[m, :] @ head_w (256, head_n) + head_b        */
#define SERL_TGEMM_EPI_PARTIAL 4          /* k-split partial products left in the workspace [(member * splits + s)][M][N] for serl_enc_finish */
#define SERL_TGEMM_EPI_LN_TANH_POLICY 3   /* ... two heads (means, log-stds) -> clipped std, u = mu + std * noise, act = tanh(u), logp */
#define SERL_TGEMM_EPI_LN_RELU_HEAD 5     /* N == 256: d = (acc + bias) [* keep_mask / keep]; C = relu(LayerNorm(d) * scale + ln_bias);
                                             head_out[m, :head_n] = C[m, :] @ head_w + head_b; optional xhat, rstd (reward classifier) */
typedef struct serl_tgemm_problem {
  const float* A; const float* B;
  int64_t sAz, sAm, sAk, sBz, sBk, sBn;
  int32_t Z;
  float* C; int64_t sCz; int32_t ldc;            /* may be NULL for the LayerNorm epilogues (activation not kept)          */
  const float* bias; int64_t sBiasZ;
  const float* ln_scale; const float* ln_bias; int64_t sLnZ;
  float* xhat; float* rstd; int64_t sXhatZ, sRstdZ;   /* optional saves for the backward pass: xhat (M, 256), rstd (M)     */
  const float* head_w; const float* head_b; int64_t sHeadWz, sHeadBz;
  float* head_out; int64_t sHeadOutZ; int32_t ld_head;  /* HEAD: (M, head_n) with row stride ld_head; POLICY: means (M, A)   */
  const float* head_w2; const float* head_b2; float* head_out2;   /* POLICY: log-std head and its raw output (M, A)        */
  const float* noise; float* act; int32_t ld_act; float* logp; float* u_out; float* std_out;   /* POLICY (Z == 1)          */
  const uint8_t* keep_mask; float keep;          /* LN_RELU_HEAD: optional (M, 256) dropout keep mask (16-byte aligned), keep probability */
} serl_tgemm_problem;
typedef struct serl_tgemm_desc {
  const serl_tgemm_problem* problems; int32_t num_problems;   /* HOST array                                                */
  int32_t M, N, K;
  int32_t epilogue, head_n;
  int32_t accumulate, reduce_z, splits;          /* splits: 0 = automatic k-split (one problem per launch when > 1)        */
  float ln_eps, std_min, std_max; int32_t deterministic;
  float* workspace; size_t workspace_bytes;      /* k-split / reduce_z partials                                           */
  int32_t* error;                                /* device int32, OR-ed with 32 if a pipeline barrier timed out             */
} serl_tgemm_desc;
int serl_tgemm_tf32(const serl_tgemm_desc* d, void* stream);

/* Batched companions of serl_tgemm_tf32 (csrc/heads_fused.cu): one launch over every problem of a step. */
#define SERL_HEADS_MAX_PROBLEMS 12
typedef struct serl_sle_problem {             /* SpatialLearnedEmbeddings (+ Dropout keep mask), vision/resnet_v1.py:81-116,352 */
  const float* feat; const float* kernel; const uint8_t* keep_mask; float* out; int32_t ld_out;
} serl_sle_problem;
int serl_sle_fwd_multi(const serl_sle_problem* problems /*host*/, int num_problems, float keep, int N, int P, int C, int F, void* stream);
typedef struct serl_sle_bwd_problem {         /* SLE kernel gradient: dkernel[p,c,f] = sum_n feat[n,p,c] * dout[n, c*8+f]              */
  const float* feat; const float* dout; int32_t ld_dout; float* dkernel;
} serl_sle_bwd_problem;
int serl_sle_bwd_multi(const serl_sle_bwd_problem* problems /*host*/, int num_problems, float* workspace, size_t workspace_bytes,
                       int N, int P, int C, int F, void* stream);
typedef struct serl_enc_finish_problem {      /* out = tanh(LayerNorm(z + bias) * scale + ln_bias), z from k-split partials or a small dense */
  const float* partials; int32_t S;           /* (S, rows, D) partial products of serl_tgemm_tf32, or NULL                      */
  const float* x; int32_t ld_x; const float* w; int32_t K;   /* else z = x (rows, K) @ w (K, D): the proprio Dense, encoding.py:65 */
  const float* bias; const float* ln_scale; const float* ln_bias;
  float* out; int32_t ld_out; float* xhat; float* rstd; int32_t D;   /* D <= 256                                                  */
} serl_enc_finish_problem;
int serl_enc_finish(const serl_enc_finish_problem* problems /*host*/, int num_problems, int rows, float eps, void* stream);
typedef struct serl_ln_bwd_problem {          /* LayerNorm + tanh backward; upstream gradient dt (+ dt2), or dq[row] * head_w[group][d] */
  const float* dt; int32_t ld_dt; const float* dt2; int32_t ld_dt2; const float* dq; const float* head_w; int64_t head_w_stride;
  const float* t; int32_t ld_t; const float* xhat; const float* rstd; const float* scale; int32_t rows_per_group; int64_t group_stride;
  float* dz; float* dy; int32_t R, D;
  int32_t dt_parts; int64_t dt_part_stride;   /* > 1: dt is the sum of dt_parts arrays (ensemble partials of serl_tgemm_tf32's PARTIAL epilogue) */
} serl_ln_bwd_problem;
int serl_layernorm_tanh_bwd_multi(const serl_ln_bwd_problem* problems /*host*/, int num_problems, void* stream);
#define SERL_SMALL_GRAD_MAX_JOBS 12
#define SERL_SMALL_GRAD_COLSUM 0              /* out_a[g][d] = sum_r x[g*rows + r][d]                     (bias gradients)         */
#define SERL_SMALL_GRAD_LN 1                  /* out_a = sum_r x*y (scale), out_b = sum_r x (bias)        (x = dy, y = xhat)        */
#define SERL_SMALL_GRAD_HEAD 2                /* out_a[g][d] = sum_r x[r][d] * y[r], out_b[g] = sum_r y[r] (x = h, y = dq: value head) */
typedef struct serl_small_grad_job {
  int32_t kind; const float* x; int64_t ld_x; const float* y; int64_t ld_y; float* out_a; float* out_b; int32_t groups, rows, D;
} serl_small_grad_job;
int serl_small_grads(const serl_small_grad_job* jobs /*host*/, int num_jobs, void* stream);

/* SpatialLearnedEmbeddings (vision/resnet_v1.py:81-116) + Dropout (resnet_v1.py:352) */
int serl_sle_fwd(const float* feat, const float* kernel, const uint8_t* keep_mask, float keep, float* out,
                 int N, int P, int C, int F, int ld_out, void* stream);
int serl_sle_bwd_kernel_grad(const float* feat, const float* dout, float* dkernel, float* workspace, size_t workspace_bytes,
                             int N, int P, int C, int F, int ld_dout, void* stream);
/* LayerNorm(eps, fast variance) + tanh, rows grouped for vmapped (ensemble) parameters (networks/mlp.py:26-31) */
int serl_layernorm_tanh_fwd(const float* z, int ld_z, const float* scale, const float* bias, int rows_per_group, int group_stride,
                            float* out, int ld_out, float* xhat, float* rstd, int R, int D, float eps, void* stream);
int serl_layernorm_tanh_bwd(const float* dt, int ld_dt, const float* t, int ld_t, const float* xhat, const float* rstd,
                            const float* scale, int rows_per_group, int group_stride, float* dz, float* dy,
                            float* dscale, float* dbias, int R, int D, void* stream);
int serl_layernorm_param_grad(const float* dy, const float* xhat, float* dscale, float* dbias, int rows_per_group, int R, int D,
                              void* stream);   /* dscale/dbias half of serl_layernorm_tanh_bwd (when it was called with NULLs) */
/* Reward classifier hidden layer (networks/reward_classifier.py:22-26): Dense -> Dropout(keep) -> LayerNorm(eps, fast variance) -> ReLU.
 * Forward (fp32 build; the 16-bit builds use SERL_TGEMM_EPI_LN_RELU_HEAD): z (R, D) = Dense output incl. bias,
 * d = keep_mask ? z / keep : 0 (keep_mask NULL: d = z), out = relu(xhat * scale + bias), optional saves xhat (R, D), rstd (R).
 * Backward (both builds): upstream gradient dt (R, D), or dlogit[r] * head_w[d] (the Dense(1) output layer, dt NULL);
 * ReLU derivative from the saved xhat * scale + bias > 0; dy (R, D) = gradient at the LayerNorm output (for the scale / bias
 * gradients: SERL_SMALL_GRAD_LN); dz (R, D) = gradient at z (dropout mask and 1/keep applied).  D <= 256. */
int serl_layernorm_relu_fwd(const float* z, int ld_z, const uint8_t* keep_mask, float keep, const float* scale, const float* bias,
                            float* out, int ld_out, float* xhat, float* rstd, int R, int D, float eps, void* stream);
/* Dropout backward in place over n elements: x = keep_mask ? x / keep : 0 */
int serl_dropout_bwd(float* x, const uint8_t* keep_mask, float keep, long long n, void* stream);
int serl_layernorm_relu_bwd(const float* dt, int ld_dt, const float* dlogit, const float* head_w, const float* xhat, const float* rstd,
                            const float* scale, const float* bias, const uint8_t* keep_mask, float keep, float* dz, float* dy,
                            int R, int D, void* stream);
int serl_colsum_f32(const float* x, float* out, int groups, int rows, int D, long long ld, int accumulate, void* stream);
int serl_copy2d_f32(const float* src, long long ld_src, float* dst, long long ld_dst, int R, int D, void* stream);
int serl_fill_f32(float* x, float v, int n, void* stream);

/* ---- SAC losses (agents/continuous/sac.py:118-234, networks/actor_critic_nets.py:230-272) -------- */
int serl_tanh_gaussian_fwd(const float* mu, const float* log_std, const float* eps, float std_min, float std_max,
                           float* act, int ld_act, float* logp, float* u_out, float* std_out, int B, int A,
                           int deterministic, void* stream);
int serl_critic_loss(const float* q, const float* q_next, const int32_t* sub, int n_sub, const float* rewards,
                     const float* masks, const float* logp_next, const float* lagrange, int backup_entropy, float gamma,
                     float grad_scale, float* target_q, float* dq, float* info /*3*/, int E, int B, void* stream);
int serl_actor_loss(const float* q, const float* logp, const float* lagrange, const float* da, int ld_da, const float* act,
                    int ld_act, const float* std, const float* log_std, const float* eps, float std_min, float std_max,
                    float grad_scale, float* dmu, float* dlogstd, float* info /*3*/, int E, int B, int A, void* stream);
/* Behaviour cloning (agents/continuous/bc.py:36-76, launcher policy utils/launcher.py:26-47: Dense -> tanh, no LayerNorm):
 * element-wise tanh forward / backward, and loss = -mean_b log N(a_b; mu_b, diag(clip(exp(log_std_b))^2)) with its gradients
 * w.r.t. mu / log_std (scaled by grad_scale / B) and info = {actor_loss, mse} * grad_scale. */
int serl_tanh_fwd(const float* z, float* out, int n, void* stream);
int serl_tanh_bwd(const float* dt, const float* t, float* dz, int n, void* stream);
int serl_bc_loss(const float* mu, const float* log_std, const float* actions, float std_min, float std_max, float grad_scale,
                 float* dmu, float* dlogstd, float* info /*2*/, int B, int A, void* stream);
int serl_temperature_loss(const float* logp, const float* lagrange, float target_entropy, float grad_scale,
                          float* dlagrange, float* info /*1*/, int B, void* stream);
/* Reward classifier loss (examples/async_cable_route_drq/train_reward_classifier.py:122-137): optax.sigmoid_binary_cross_entropy(x, y).mean()
 * = mean(relu(x) - x*y + log1p(exp(-|x|))) over the train logits x (B), labels y (B);
 * dlogit = grad_scale * (sigmoid(x) - y) / B; info[0] = loss, info[1] = mean((sigmoid(x_eval) >= 0.5) == y) over the eval
 * logits (train=False pass, pre-update parameters), both * grad_scale.  One CTA, fixed-order reduction. */
int serl_bce_logits_loss(const float* logits, const float* eval_logits, const float* labels, int B, float grad_scale,
                         float* dlogit, float* info /*2*/, void* stream);

/* Stride-1 3x3 convolution + GroupNorm(4 groups) [+ residual] [+ ReLU] in one kernel (vision/resnet_v1.py:129-156: the
   ResNetBlock body after / including each 3x3 conv).  An image's accumulators stay in tensor memory until its statistics are
   complete, so no raw conv output and no normalisation pass ever touch HBM:
       y = [relu]( GN(conv3x3(x, w); gamma, beta) [+ res | + GN_res(res)] )
   x (N,H,W,Ci), res / y (N,H,W,Co) 16-bit NHWC; w packed [Co][9*Ci] K-major ((kh,kw,ci) order); out_f32 (N,H,W,Co) replaces y
   for the last block.  res_stats (N,4,2) + res_gamma/res_beta: the residual is a RAW projection-conv output whose own
   GroupNorm is applied on the fly.  Shapes: the four ResNet-10 block shapes at 128x128 input (H=W in {32,16,8,4}, Ci=Co). */
typedef struct serl_conv3x3_res_desc {
  const void* x; const void* w; void* y; float* out_f32; const void* res;
  const float* gamma; const float* beta;
  const float* res_stats; const float* res_gamma; const float* res_beta;
  int32_t* error;
  int32_t N, H, W, Ci, Co, relu, fmt;
  float eps;
} serl_conv3x3_res_desc;
int serl_conv3x3_res_h16(const serl_conv3x3_res_desc* d, void* stream);

/* Head of ResNetBlock_1..3 in one kernel (vision/resnet_v1.py:139-154): x (N,2Wo,2Wo,Ci) ->
       y = relu(GN(conv3x3 stride 2 SAME(x, w); gamma, beta))            (N,Wo,Wo,Co), Co = 2 Ci
       r = GN(conv1x1 stride 2(x, w_proj); gamma_proj, beta_proj)        (N,Wo,Wo,Co)   (the block's residual branch, normalised)
   w packed [Co][9*Ci], w_proj [Co][Ci], K-major 16-bit.  Wo in {16, 8, 4} (Co = 128, 256, 512). */
typedef struct serl_conv3x3s2_res_desc {
  const void* x; const void* w; const void* w_proj; void* y; void* r;
  const float* gamma; const float* beta; const float* gamma_proj; const float* beta_proj;
  int32_t* error;
  int32_t N, Wo, Ci, Co, fmt;
  float eps;
} serl_conv3x3s2_res_desc;
int serl_conv3x3s2_res_h16(const serl_conv3x3s2_res_desc* d, void* stream);

/* ---- optimizer (common/common.py:124-168, common/optimizers.py:6-56) --------------------------- */
typedef struct serl_adam_desc {
  float* params; float* target; float* m; float* v; const float* grad;
  int32_t n;
  int32_t seg_end[3];        /* flat layout: group 0 = critic tx, 1 = actor tx, 2 = temperature tx */
  int32_t live[3];           /* network updated this call (else its gradient is zero)             */
  int32_t* counts;           /* device int32[3]: optax counts, incremented by the call            */
  float lr[3]; int32_t warmup[3];
  float b1, b2, eps, tau;
  int32_t polyak;            /* soft target update after the step                                 */
  float* lr_out;             /* optional device float[3]                                          */
  /* Flat-buffer extras (serl_b200/params.py): `n` counts parameter slots only; indices in
     [seg_end[0], seg_end[0] + gap) hold no parameter (info scalars of the gradient buffer) and are
     skipped.  Leaves in [aux_lo, aux_hi) are updated by TWO transforms (reference
     common/common.py:136-168: the proprio encoder gets gradients from the critic loss AND from the
     actor loss, common/encoding.py:48-70): group 0 through grad/m/v[i] and group 1 (the actor tx)
     through grad/m/v[i + aux_off]; the two updates are summed before they are applied.            */
  int32_t gap, aux_lo, aux_hi, aux_off;
} serl_adam_desc;
int serl_adam_polyak(const serl_adam_desc* d, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SERL_B200_H_ */
