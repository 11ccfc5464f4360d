/*
 * hi3d_b200.h -- C ABI of libhi3d_b200.so: the B200 (sm_100a) kernels behind the Hi3D denoising hot path.
 *
 * Boundary (SURVEY.md 8b): the reference is pure Python/PyTorch; its "FFI" for this path is the set of
 * ATen / cuDNN / cuBLAS / xformers calls its nn.Modules make.  Each entry point below replaces one such
 * call site (cited as reference file:line, relative to the Hi3D-Official tree) and is what a maintainer
 * of the reference would bind with ctypes/cffi (stub shown in INTEGRATION.md).
 *
 * Conventions
 *   - plain pointers + sizes; no torch types.  All pointers are DEVICE pointers unless noted.
 *   - activations are fp16, channels-last: a feature map is [N, H, W, C] == a token matrix [N*H*W, C];
 *     frames of a clip are consecutive samples, n = b*T + t (reference "(b t)" order, video_model.py:71).
 *   - every call only enqueues work on `stream` (a cudaStream_t passed as void*): no allocation, no
 *     host synchronisation, safe to capture in a CUDA graph.  Workspaces are caller-owned.
 *   - return 0 on success, negative on error; hi3d_last_error() returns a thread-local message.
 */
#ifndef HI3D_B200_H_
#define HI3D_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HI3D_MAX_SEGS 24
#define HI3D_MAX_PEERS 16   /* ranks of one frame-sharded video (16 frames) */

/* library ------------------------------------------------------------------------------------ */
int hi3d_abi_version(void);
const char* hi3d_last_error(void);
/* Number of kernels this library has launched since load (for bench.py's `gpu_launches`). */
int64_t hi3d_launch_count(void);
/* sm count etc. of the current device (cached).  Returns 0 or negative error. */
int hi3d_device_info(int* sm_count, int* cc_major, int* cc_minor, int* max_smem_optin);

/* ---------------------------------------------------------------------------------------------
 * Implicit-GEMM engine.  out[M, N] = epilogue( A[M, K] * W[N, K]^T )
 *
 * A is never materialised: its K axis is a list of segments, each a (tap, channel-range) view of an
 * NHWC fp16 tensor.  This one entry point replaces, in the reference:
 *   nn.Linear                      attention.py:272-278 (to_q/k/v/out), :90 (GEGLU proj), :109 (ff out),
 *                                  video_attention.py:221-223 (time_pos_embed), openaimodel.py:286 (emb)
 *   nn.Conv2d 3x3 s1/s2, 1x1       openaimodel.py:135,192,260,297,314; model.py:63,82,110,117,127
 *   nearest-x2 + Conv2d            openaimodel.py:154-156; model.py:67-70     (ups = 1)
 *   F.pad(0,1,0,1) + Conv2d s2 p0  model.py:84-88                              (taps dy,dx in {0,1,2})
 *   nn.Conv3d (3,1,1)              openaimodel.py:260,297 with dims=3 via video_model.py:42-55 (mode 2)
 *   th.cat([h, hs.pop()], 1)       video_model.py:491  (two segments per tap = virtual concat)
 *   skip_connection 1x1 / nin_shortcut   openaimodel.py:314,354; model.py:127,149 (extra K segments)
 * and in the epilogue: + bias, + emb[:, :, None, None] (openaimodel.py:352), residual adds
 * (attention.py:551-572), GEGLU x*gelu(gate) (attention.py:92-94), AlphaBlender (util.py:358-369).
 * --------------------------------------------------------------------------------------------- */
typedef struct {
  const void* src;   /* fp16 NHWC source tensor                                            */
  int32_t ld;        /* elements between consecutive pixels/rows of src (its channel count) */
  int32_t c_off;     /* first channel of the segment                                        */
  int32_t C;         /* channels in the segment; multiple of 64                             */
  int32_t dy, dx;    /* spatial tap offset in (upsampled) input coordinates                 */
  int32_t dt;        /* temporal tap offset in frames (mode 2)                              */
} hi3d_seg;

enum { HI3D_ROWS_PLAIN = 0, HI3D_ROWS_CONV2D = 1, HI3D_ROWS_TEMPORAL = 2 };
enum { HI3D_ACT_NONE = 0, HI3D_ACT_SILU = 1, HI3D_ACT_GEGLU = 2 };

typedef struct {
  int32_t M, N, K;          /* K == sum of seg[i].C; N multiple of 8                                   */
  int32_t mode;             /* HI3D_ROWS_*                                                             */
  int32_t Ho, Wo;           /* CONV2D: output H, W (M == Nimg*Ho*Wo).  TEMPORAL: Ho*Wo = rows per frame */
  int32_t Hs, Ws;           /* CONV2D: source H, W (before the optional x2 nearest upsample)           */
  int32_t stride;           /* CONV2D: 1 or 2                                                          */
  int32_t ups;              /* CONV2D: 1 -> taps address the x2 nearest-upsampled source               */
  int32_t T;                /* TEMPORAL: frames per clip                                               */
  int32_t out_up;           /* CONV2D: 1 -> rows index an (n, y, x) grid of Ho x Wo but are WRITTEN to the x2 grid at
                               (2y + out_py, 2x + out_px): one parity class of nearest-x2 + conv3x3, which is a 2x2
                               conv on the source grid with pre-summed taps (4 launches, 4/9 of the FLOPs)       */
  int32_t out_py, out_px;
  int32_t Tin, t_off;       /* TEMPORAL: frames per clip in the SOURCE tensors and frame offset of output frame 0 in it
                               (0, 0 -> Tin = T).  Frame-sharded runs read a haloed [B, T_local + 2, HW, C] buffer:
                               Tin = T + 2, t_off = 1; taps that fall outside [0, Tin) read zeros.            */
  int32_t nseg;
  hi3d_seg seg[HI3D_MAX_SEGS];
  const void* W;            /* fp16 [N, K], K contiguous, K ordered as the segments                    */
  const float* bias;        /* [N] or NULL                                                             */
  const void* rowbias;      /* fp16 [R, rb_ld] or NULL; row r = (m / rb_div) % rb_mod                  */
  int32_t rb_div, rb_mod, rb_ld;
  int32_t act;              /* HI3D_ACT_*; GEGLU: W rows interleaved (value, gate), output width N/2   */
  const void* residual;     /* fp16 [M, res_ld] or NULL, added after the activation                    */
  int32_t res_ld;
  const void* blend_x;      /* fp16 [M, blend_ld] or NULL: out = alpha*blend_x + (1-alpha)*value       */
  int32_t blend_ld;
  float alpha;
  void* out;                /* fp16 [M, out_ld]                                                        */
  int32_t out_ld;
  /* GroupNorm statistics of the OUTPUT tensor, produced by the epilogue (the "GN-stats half" of the fused
   * GroupNorm+SiLU+conv of openaimodel.py:257-261,292-305: the consumer of this tensor is a GroupNorm, whose separate
   * statistics pass -- one full read of the tensor -- disappears).  gn_stats: fp32 [n_images, N / gn_unit, 2], (sum, sum of
   * squares) of the stored fp16 values per image and per unit of gn_unit consecutive channels, ACCUMULATED with atomics (the
   * caller zeroes it); image of a row = (row of the Ho x Wo / HW GEMM grid) / gn_rows.  Units, not the 32 groups, because a
   * consumer may normalise the channel concat of two tensors (video_model.py:491) whose groups straddle the boundary;
   * gn_unit divides every channels-per-group value of the network (model_channels / 32).  NULL = off. */
  float* gn_stats;
  int32_t gn_unit;
  int32_t gn_rows;
} hi3d_gemm_params;

int hi3d_gemm(const hi3d_gemm_params* p, void* stream);
/* Same contract on the Blackwell-native engine (persistent kernel, TMA operand staging, tcgen05.mma with TMEM
 * accumulators, CTA pairs on long-K shapes): the production path.  Geometries it does not cover (N < 32, unaligned row
 * bias, > 4 distinct A sources, ...) are forwarded to hi3d_gemm, with identical results.
 * Environment (experiments only, read once per process): HI3D_TC5_PAIR=0|1 forces single-CTA / CTA-pair tiles,
 * HI3D_TC5_DBG=<bit mask> disables parts of the kernel for bottleneck measurements (results are then meaningless). */
int hi3d_gemm_tc5(const hi3d_gemm_params* p, void* stream);
/* Test hook: -1 = automatic choice between single-CTA and CTA-pair (cta_group::2, 256-row) tiles (default, or the value of
 * HI3D_TC5_PAIR at first use), 0 = always single CTA, 1 = always CTA pairs.  Process-wide; the parity tests run every
 * geometry under both settings (no reference counterpart: the reference's cuDNN / cuBLAS pick their own tiles). */
int hi3d_gemm_tc5_set_pair_mode(int mode);
/* Deterministic GroupNorm statistics: hi3d_gemm / hi3d_gemm_tc5 with p->gn_stats produced without float atomics, in an order
 * that depends on the shapes and the tile geometry only, so that the same inputs give the same bits on every run.  gn_stats is
 * OVERWRITTEN (no zeroing needed).  `partials` is caller-owned fp32 scratch of partials_floats >=
 * hi3d_groupnorm_partials_floats(n_images, output rows per image, N, gn_unit) floats; it is dead once the statistics are
 * complete and may be reused by the next producer on the same stream.  How the table is produced:
 *   - hi3d_gemm_tc5_det, specialised GroupNorm epilogues, gn_unit == 4 or >= 8, and every 32-row warp block inside one image
 *     (PLAIN: gn_rows % 32 == 0; CONV2D: tile patch of >= 32 pixels per image; TEMPORAL: >= 32 pixels per frame): each
 *     epilogue warp STORES its per-octet partials into its own slot (one slot per image, 32-row block and 8-channel octet;
 *     the four parity-class launches of an up-conv have separate slots) and hi3d_groupnorm_fold sums them after the launch
 *     (after the out_py = out_px = 1 launch of an up-conv);
 *   - otherwise (narrower units, several images inside a warp -- test-sized models only -- the generic epilogue, or the
 *     mma.sync engine) the GEMM runs without epilogue statistics and hi3d_groupnorm_unit_stats_det reads the stored tensor
 *     (after the last parity launch of an up-conv; out_ld must equal N).
 * Without gn_stats they are hi3d_gemm / hi3d_gemm_tc5. */
int hi3d_gemm_det(const hi3d_gemm_params* p, float* partials, int64_t partials_floats, void* stream);
int hi3d_gemm_tc5_det(const hi3d_gemm_params* p, float* partials, int64_t partials_floats, void* stream);
/* Test / tuning hook: epilogue warps of the specialised bias-only and GEGLU epilogues: -1 = automatic (16 when K <= 640, the
 * GEMMs whose epilogue is the bound), 8 or 16 forced.  Process-wide; default from HI3D_TC5_EW. */
int hi3d_gemm_tc5_set_epilogue_warps(int warps);

/* Tiny channel counts (UNet input 8|17 ch, VAE image 3 ch / latent 4 ch) are zero-padded to 64 channels by
 * hi3d_sampler_pre / hi3d_nchw_to_nhwc so that the same engine serves input_blocks.0.0 (video_model.py:186-191),
 * encoder.conv_in (model.py:517) and decoder.conv_in (model.py:654); tiny C_out (4 | 8 | 3) is padded to 8. */

/* ---------------------------------------------------------------------------------------------
 * Normalisation
 * --------------------------------------------------------------------------------------------- */
/* GroupNorm(32 groups) [+ SiLU] over `rows_per_sample` consecutive rows x (C/32) channels, on the virtual
 * channel-concat of up to two NHWC fp16 sources (x1: C1 channels, x2: C2 channels or NULL).
 * Replaces GroupNorm32 (util.py:274-276; eps 1e-5; temporal ResBlock: rows_per_sample = T*H*W, i.e. the
 * reduction over (C/32, T, H, W) of video_model.py:71-76), Normalize (attention.py:125-128, model.py:52-55;
 * eps 1e-6) and the following nn.SiLU / x*sigmoid(x).  Two launches: partial sums then apply.
 * ws: fp32 workspace of hi3d_groupnorm_ws_floats(n_samples) floats. Output y: fp16 [rows, C1+C2]. */
int64_t hi3d_groupnorm_ws_floats(int n_samples);
int hi3d_groupnorm_silu(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                        const float* gamma, const float* beta, float eps, int apply_silu, void* y, float* ws,
                        void* stream);

/* The two halves of hi3d_groupnorm_silu, exposed for frame-sharded runs where the temporal ResBlock's GroupNorm reduces
 * over (C/32, T, H, W) with T split over GPUs (SURVEY F9): `sums` fp32 [n_samples, 32, 2] = (sum, sum of squares) of the
 * local rows; the host all-reduces them over ranks and passes count_rows = the GLOBAL rows per sample.  y may be a
 * haloed buffer: sample n starts at row n * y_sample_rows + y_row_off (0, 0 = dense). */
int hi3d_groupnorm_sums(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample, float* sums,
                        float* ws, void* stream);
int hi3d_groupnorm_apply(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                         const float* sums, int64_t count_rows, const float* gamma, const float* beta, float eps,
                         int apply_silu, void* y, int64_t y_sample_rows, int64_t y_row_off, void* stream);

/* hi3d_groupnorm_apply for frame-sharded runs with the one-frame halo exchange of the temporal (3,1,1) conv fused into its
 * stores: y = [n, T_local + 2, frame_rows, C] (y_sample_rows = (T_local + 2) * frame_rows, y_row_off = frame_rows); the first
 * local frame is also stored into the trailing halo slot of `y_prev_rank` (the same buffer of the rank holding the previous
 * frames, mapped through hi3d_symm_open) and the last local frame into the leading slot of `y_next_rank`; NULL at the clip
 * boundaries: the local halo slot is then zero-filled (the Conv3d zero padding, openaimodel.py:252-261).  A hi3d_peer_exchange must
 * separate this launch from the conv that reads the halo slots. */
/* The consumer side of hi3d_gemm_params::gn_stats: GroupNorm(32)[+SiLU] whose statistics come from the per-image, per-unit
 * (sum, sumsq) tables written by the GEMM epilogues that produced x1 / x2 (stats1: fp32 [n_images, C1/unit, 2], stats2
 * likewise or NULL) instead of a statistics pass over the tensor: ONE launch per GroupNorm.  Sample n spans images
 * [n*imgs_per_sample, (n+1)*imgs_per_sample) -- 1 for the spatial GroupNorm32, T for the temporal ResBlock's reduction over
 * (C/32, T, H, W) (video_model.py:71-76).  Other arguments as hi3d_groupnorm_apply_halo (frame_rows = 0: dense output). */
int hi3d_groupnorm_apply_stats(const void* x1, int C1, const float* stats1, const void* x2, int C2, const float* stats2,
                               int unit, int n_samples, int64_t rows_per_sample, int imgs_per_sample, int64_t count_rows,
                               const float* gamma, const float* beta, float eps, int apply_silu, void* y, int64_t y_sample_rows,
                               int64_t y_row_off, void* y_prev_rank, void* y_next_rank, int64_t frame_rows, void* stream);
/* Unit statistics of an existing tensor (same table as hi3d_gemm_params::gn_stats, accumulated): for tensors not produced
 * by an epilogue that can do it (the mma.sync engine uses this internally), and unit tables -> group sums
 * fp32 [n_samples, 32, 2] (what the frame-sharded temporal GroupNorm all-reduces over ranks). */
int hi3d_groupnorm_unit_stats(const void* x, int C, int n_images, int64_t rows_per_image, int unit, float* stats, void* stream);
int hi3d_groupnorm_group_sums(const float* stats1, int C1, const float* stats2, int C2, int unit, int n_samples,
                              int imgs_per_sample, float* sums, void* stream);

int hi3d_groupnorm_apply_halo(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                              const float* sums, int64_t count_rows, const float* gamma, const float* beta, float eps,
                              int apply_silu, void* y, int64_t y_sample_rows, int64_t y_row_off, void* y_prev_rank,
                              void* y_next_rank, int64_t frame_rows, void* stream);

/* Deterministic GroupNorm statistics: the same contracts without float atomics, every sum in an order fixed by the shapes
 * (and launch geometry) alone, so the same inputs give bit-identical results run after run.  They are what a launch plan
 * uses when torch.use_deterministic_algorithms(True) or HI3D_DETERMINISTIC=1 is in effect.  Bit-identity holds for one
 * build on one GPU type and one configuration; a different tile geometry, engine or sharding may round differently.
 *   hi3d_groupnorm_silu_det / hi3d_groupnorm_sums_det: as hi3d_groupnorm_silu / _sums (same workspace).
 *   hi3d_groupnorm_group_sums_det: as hi3d_groupnorm_group_sums.
 *   hi3d_groupnorm_unit_stats_det: the unit table of x, OVERWRITTEN (not accumulated): one partials slot per (image, chunk),
 *     stored by the statistics pass, then hi3d_groupnorm_fold.  `partials` = fp32 scratch of partials_floats >=
 *     hi3d_groupnorm_partials_floats(n_images, rows_per_image, C, unit) floats.
 *   hi3d_groupnorm_partials_floats: scratch floats any deterministic producer of an [n_images, C / unit, 2] table over
 *     rows_per_image output rows per image needs (0 on bad arguments).
 *   hi3d_groupnorm_fold: stats[n, u, :] = sum over the blocks_per_image slots of image n of a partials table, in fp64, in a
 *     fixed order, stored as fp32 (overwrites stats).  octets = 0: slots [n_images, blocks_per_image, C / unit, 2] (the
 *     statistics pass); octets = 1: slots [n_images, blocks_per_image, C / 8, 4] = (sum, sumsq) of the first unit an
 *     8-channel octet touches, then of the next one (the tc5 epilogue; unit == 4 or >= 8). */
int hi3d_groupnorm_silu_det(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample,
                            const float* gamma, const float* beta, float eps, int apply_silu, void* y, float* ws, void* stream);
int hi3d_groupnorm_sums_det(const void* x1, int C1, const void* x2, int C2, int n_samples, int64_t rows_per_sample, float* sums,
                            float* ws, void* stream);
int hi3d_groupnorm_group_sums_det(const float* stats1, int C1, const float* stats2, int C2, int unit, int n_samples,
                                  int imgs_per_sample, float* sums, void* stream);
int hi3d_groupnorm_unit_stats_det(const void* x, int C, int n_images, int64_t rows_per_image, int unit, float* stats,
                                  float* partials, int64_t partials_floats, void* stream);
int64_t hi3d_groupnorm_partials_floats(int n_images, int64_t rows_per_image, int C, int unit);
int hi3d_groupnorm_fold(const float* partials, int n_images, int blocks_per_image, int octets, int C, int unit, float* stats,
                        void* stream);

/* LayerNorm over the last dim C (<= 2560, multiple of 8) of [M, C] fp16 (+ optional broadcast add before the norm:
 * x + addvec[((m / add_div) % add_mod), :], the `x_mix = x + emb` of video_attention.py:286-287).
 * Replaces nn.LayerNorm at attention.py:520-522, video_attention.py:51,79,93-94.  y fp16 [M, C]. */
int hi3d_layernorm(const void* x, const void* addvec, int add_div, int add_mod, int64_t M, int C, const float* gamma,
                   const float* beta, float eps, void* y, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Attention
 * --------------------------------------------------------------------------------------------- */
/* Spatial self-attention core, head dim 64: softmax(Q K^T * scale) V per (image, head).
 * qkv: fp16 [n_img*L, 3*C] with q | k | v column blocks, heads contiguous (C = heads*64); out fp16 [n_img*L, C].
 * Replaces F.scaled_dot_product_attention / xformers.memory_efficient_attention at attention.py:334,427-439. */
int hi3d_attention_d64(const void* qkv, int n_img, int L, int heads, float scale, void* out, void* stream);
/* same contract on tcgen05 / TMEM / TMA (S and P*V accumulators in tensor memory, P fed back from TMEM);
 * sequences that are not a multiple of 128 keys are forwarded to hi3d_attention_d64. */
int hi3d_attention_d64_tc5(const void* qkv, int n_img, int L, int heads, float scale, void* out, void* stream);
/* Tuning / test hook of hi3d_attention_d64_tc5: `quarters` / 4 of the softmax exponentials (0 .. 4; 3 and 4 only with
 * variants >= 2) are evaluated on the FMA pipe (range reduction + cubic polynomial, relative error 7.5e-5 before the fp16
 * rounding of P) instead of the MUFU pipe.  Process-wide; default from HI3D_FMHA_EMU, else the measured best. */
int hi3d_attention_tc5_set_exp_emulation(int quarters);
/* Kernel variant of hi3d_attention_d64_tc5: 0 = eight softmax warps share one score tile, reference maximum and P barrier
 * per CTA; 1 = the 128 keys of a tile are two independent 64-key pipelines (own score / P columns, accumulator, barriers and
 * per-row state), merged once at the end; 2 = 1 with the register-lean softmax loop (scores read in 16-column chunks, P
 * stored once the half-tile is accepted by its row sum); 3 = 2 + the MMA warp serves whichever half is ready; 4 = 2 + strict
 * turns between the halves; 5 = 2 with clock stamps (tools only); 6 = 2 with the scores of a half issued as two 32-key blocks,
 * the first one ahead of P V.  Process-wide; default from HI3D_FMHA_VARIANT, else the
 * measured best. */
int hi3d_attention_tc5_set_variant(int variant);
/* tools/fmha_timeline.py: device buffer of 128 int64 that variant 5 fills with clock64 stamps of one CTA; NULL = off. */
int hi3d_attention_tc5_set_debug_buffer(void* buf);

/* Temporal self-attention core over the frame axis (T <= 16), head dim 64, for every (clip, pixel, head):
 * token row of (b, t, s) is (b*T + t)*S + s -- the "(b t) s c -> (b s) t c" rearrange of
 * video_attention.py:114,137-139 is done by addressing, never materialised.
 * qkv fp16 [B*T*S, 3*C]; out fp16 [B*T*S, C].  Replaces attn1 core at video_attention.py:125. */
int hi3d_temporal_attention_d64(const void* qkv, int B, int T, int S, int heads, float scale, void* out,
                                void* stream);

/* Frame-sharded form (SURVEY 8e; the reference has no multi-GPU inference, README.md:56-64): rank r owns frames
 * [r*T_local, (r+1)*T_local) of every clip in its own qkv / out buffers (layout as above with T = T_local) and computes
 * pixel strip r of all T_local*world frames: q|k|v rows of the other ranks' frames are READ from `qkv_of_rank[owner]` and the
 * output rows of their frames are STORED into `out_of_rank[owner]` (device pointers of the peers' buffers mapped with
 * hi3d_symm_open; entry [rank] = the local buffers).  One hi3d_peer_exchange before (all q|k|v written) and one after (all
 * outputs stored) order it against the producing / consuming GEMMs. */
int hi3d_temporal_attention_d64_sharded(void* const* qkv_of_rank, void* const* out_of_rank, int rank, int world, int B,
                                        int T_local, int S, int heads, float scale, void* stream);

/* VAE mid-block attention (AttnBlock, model.py:180-201; xformers path model.py:204-265): ONE head of dimension 512,
 * softmax(q k^T * scale) v per image with scale = 512^-0.5, as a flash-attention kernel (tcgen05 / TMEM / TMA): fp32
 * scores and softmax, no L x L matrix in memory.  qkv: fp16 [n_img*L, 1536] = q | k | v column blocks (the three 1x1 convs as
 * one GEMM); out fp16 [n_img*L, 512].  L must be a multiple of 128 ((H/8)*(W/8) at every Hi3D size). */
int hi3d_attention_d512_tc5(const void* qkv, int n_img, int L, float scale, void* out, void* stream);

/* Row softmax in place on fp16 [rows, L] (scores * scale), and 2-D transpose [R, Cc] -> [Cc, R] (fp16):
 * building blocks of the VAE single-head d=512 attention (model.py:180-195) on top of hi3d_gemm. */
int hi3d_softmax_rows(void* s, int64_t rows, int L, float scale, void* stream);
int hi3d_transpose(const void* in, int R, int Cc, int in_ld, void* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Sampler-side fused elementwise kernels (EulerEDMSampler / Denoiser / LinearPredictionGuider)
 * --------------------------------------------------------------------------------------------- */
/* timestep_embedding (util.py:207-231): t fp32 [n] -> fp16 [n, dim] = [cos | sin]. */
int hi3d_timestep_embedding(const float* t, int n, int dim, float max_period, void* out, void* stream);

/* Build the UNet input for one CFG-batched step: prepare_inputs (guiders.py:88-99) + Denoiser c_in scaling
 * (denoiser.py:33-37) + OpenAIWrapper concat (wrappers.py:27) + NCHW->NHWC fp16.
 * x fp32 NCHW [F, Cx, H, W]; sigma fp32 [F]; concat_uc / concat_c fp16-or-fp32 NCHW [F, Cc, H, W] (concat_uc may be
 * NULL == zeros); out fp16 NHWC [2F, H, W, Cpad] (channels [x*c_in | concat | 0-pad]); first F samples = uc half.
 * c_noise_out (optional) fp32 [2F] receives c_noise = 0.25*ln(sigma) (denoiser_scaling.py:58), the UNet `timesteps`. */
int hi3d_sampler_pre(const float* x, const float* sigma, const void* concat_uc, const void* concat_c,
                     int concat_is_fp32, int F, int Cx, int Cc, int H, int W, int Cpad, void* out, float* c_noise_out,
                     void* stream);

/* Finish the step: denoised = net*c_out + x*c_skip per half (denoiser.py:36-39), CFG combine with the per-frame
 * scale (guiders.py:78-86), d = (x - denoised)/sigma and Euler update x += d*(sigma_next - sigma)
 * (sampling.py:99-103, sampling_utils.py:34).  net fp16 NHWC [2F, H, W, net_ld] (first Cx channels used);
 * x fp32 NCHW [F, Cx, H, W] updated in place (x_out may alias x); scale fp32 [T] (frame t = f % T);
 * denoised_out optional fp32 NCHW [F, Cx, H, W] (the guided D(x, sigma), for teacher-forced parity checks). */
int hi3d_sampler_post(const void* net, int net_ld, const float* x, const float* sigma, const float* sigma_next,
                      const float* scale, int T, int F, int Cx, int H, int W, float* x_out, float* denoised_out,
                      void* stream);

/* Solver algebra of the multi-evaluation samplers on the fp32 sampler state (SURVEY 8f N4): out = sum_k c_k[f] * x_k, up to four
 * terms (x1..x3 may be NULL), fp32 NCHW tensors of F samples x per_sample values, coefficients fp32 [F] on the device.
 * HeunEDMSampler (sampling.py:236-254): x + dt/2 (d + d') with d = (x - D)/sigma, d' = (x_e - D')/sigma'
 *   = (1 + dt/(2 sigma)) x - dt/(2 sigma) D + dt/(2 sigma') x_e - dt/(2 sigma') D'.
 * DPMPP2MSampler (sampling.py:305-379): (sigma'/sigma) x - expm1(-h) ((1 + 1/(2r)) D - 1/(2r) D_old). */
int hi3d_sampler_lincomb4(float* out, const float* x0, const float* x1, const float* x2, const float* x3, const float* c0,
                          const float* c1, const float* c2, const float* c3, int F, int64_t per_sample, void* stream);

/* Stage-2 re-noise blend (pipeline_i2v_eval_v02.py:131-132): lat = lat*(1-a) + (init*sigma + z)*a, fp32. */
int hi3d_renoise_blend(float* lat, const float* init, const float* z, float alpha, float sigma, int64_t n,
                       void* stream);

/* Layout / dtype helpers: NCHW (fp32 or fp16) -> NHWC fp16 with channel padding, and NHWC fp16 -> NCHW fp32/fp16
 * (first C channels), used at the VAE / latent boundaries (autoencoder.py:468-505, diffusion.py:117-150). */
int hi3d_nchw_to_nhwc(const void* in, int in_is_fp32, int N, int C, int H, int W, int Cpad, float scale, void* out,
                      void* stream);
int hi3d_nhwc_to_nchw(const void* in, int in_ld, int N, int C, int H, int W, float scale, void* out, int out_is_fp32,
                      void* stream);

/* DiagonalGaussianDistribution.sample / mode (distributions.py:24-41,71) * scale_factor (diffusion.py:149):
 * moments fp16 NHWC [N, H, W, ld] (mean = ch 0..C-1, logvar = ch C..2C-1), noise fp32 NCHW or NULL (mode),
 * out fp32 NCHW [N, C, H, W]. */
int hi3d_gaussian_sample(const void* moments, int ld, const float* noise, int N, int C, int H, int W, float scale,
                         float* out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Peer memory for the frame-sharded step (one process per GPU; SURVEY 8e).  No reference counterpart.
 * --------------------------------------------------------------------------------------------- */
/* Symmetric buffers: hi3d_symm_alloc = cudaMalloc + zero fill + cudaIpcGetMemHandle (handle64: 64 bytes the host ships to
 * the other ranks, e.g. with torch.distributed.all_gather_object); hi3d_symm_open maps a peer's buffer into this process
 * (cudaIpcOpenMemHandle, enabling peer access); hi3d_symm_close / hi3d_symm_free undo them. */
int hi3d_symm_alloc(int64_t bytes, void** ptr, void* handle64);
int hi3d_symm_open(const void* handle64, void** ptr);
int hi3d_symm_close(void* ptr);
int hi3d_symm_free(void* ptr);
/* Size of one rank's exchange area (flags + payload slots + epoch word) for hi3d_peer_exchange. */
int64_t hi3d_peer_xchg_bytes(int world);
/* One exchange point of the sharded step, a single-CTA kernel on `stream`: every rank announces a new epoch in its slot of
 * every peer's flag array and waits until all peers have announced it -- everything the ranks stored into each other's
 * buffers before this point is visible after it.  With n > 0 (<= 1024) it is also an all-reduce: out[j] = sum over ranks of
 * payload[j] in rank order (the [B, 32, 2] partial sums of the temporal GroupNorm, video_model.py:71-76).  xchg[r] = rank
 * r's exchange area (zero-initialised symmetric memory); every rank must issue the same sequence of exchanges. */
int hi3d_peer_exchange(void* const* xchg, int rank, int world, const float* payload, int n, float* out, void* stream);

/* One-time weight packing (device -> device), the C twin of hi3d_official_b200/pack.py for hosts without torch:
 * reference layouts as stored in the checkpoints -- nn.Linear [Co, Ci] (taps = 1; attention.py:269-278, 87-113),
 * Conv2d OIHW (taps = kh*kw; openaimodel.py:107-207, 263-304, model.py:67-151), Conv3d (Co, Ci, 3, 1, 1) (taps = 3;
 * video_model.py:45-60) -- into the fp16 [cout_pad, taps * cin_pad] K-major matrix of hi3d_gemm (K ordered (tap, ci),
 * zero padded).  geglu_interleave: rows of the GEGLU projection [value ; gate] are interleaved (value_j, gate_j).
 * hi3d_pack_bias: fp32 [n_pad] (b may be NULL -> zeros).  Caller owns all buffers. */
int hi3d_pack_weight(const void* w, int w_is_fp32, int Co, int Ci, int taps, int cin_pad, int cout_pad,
                     int geglu_interleave, void* out, void* stream);
int hi3d_pack_bias(const void* b, int b_is_fp32, int n, int n_pad, int geglu_interleave, float* out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HI3D_B200_H_ */
