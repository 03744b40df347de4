/* vc_b200.h -- C ABI of libvc_b200.so: the sm_100a kernels behind ViewCrafter's DDIM-denoise hot path.
 *
 * Boundary contract (SURVEY.md 8b): the reference has no FFI of its own on this path -- its "plugin API" is the
 * Python class surface (DDIMSampler.sample / UNetModel.forward / AutoencoderKL.decode).  The Python mirror of
 * those classes lives in viewcrafter_b200/{ddim,unet,autoencoder}.py and binds THIS library with ctypes
 * (viewcrafter_b200/_lib.py); a maintainer of the reference would add the same ctypes stub (INTEGRATION.md).
 *
 * Conventions: every entry point returns 0 on success, non-zero on failure (vc_last_error() holds the text);
 * all pointers are DEVICE pointers borrowed from the caller (torch storage) unless stated otherwise; `stream`
 * is a cudaStream_t passed as void*; activations are channels-last fp16 ("rows x channels", row = pixel/token);
 * parameters that the reference keeps in fp32 (norm scales, biases) stay fp32.  No call synchronises the device.
 *
 * Each declaration cites the reference code it replaces (paths relative to the upstream repo root).
 */
#ifndef VC_B200_H
#define VC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VC_B200_ABI_VERSION 7

int vc_abi_version(void);
const char* vc_last_error(void);
/* number of kernel launches issued by this library since the last vc_reset_launch_count() (bench "gpu_launches") */
long long vc_launch_count(void);
void vc_reset_launch_count(void);

/* ---- tensor-core tap-GEMM: every nn.Linear / nn.Conv2d(3x3,1x1) / nn.Conv3d(3,1,1) on the path -------------
 * replaces: torch conv2d/conv3d/linear calls in lvdm/modules/networks/openaimodel3d.py:154,179,191,255-266,
 *           lvdm/modules/attention.py:52-55,71-72,418-422,435-439, lvdm/modules/networks/ae_modules.py:157-188
 * out[row, n] = sum_tap sum_k A[row shifted by tap, k] * w[tap*N + n, k]  (+bias) (GEGLU) (+res)
 */
typedef struct vc_gemm_desc {
  const void* a;   int32_t lda;      /* fp16 A, logical (K, X, Y, Z), row pitch lda elements            */
  const void* a2;  int32_t lda2;     /* optional second K-slab (channel concat), NULL if unused          */
  int32_t X, Y, Z;                   /* spatial extents; plain GEMM: X = M rows, Y = Z = 1               */
  int32_t bx, by;                    /* 128-row tile = bx * by pixels (by > 1 requires bx == X)          */
  int32_t K, K1;                     /* reduction per tap; K1 = channels served by `a` (== K if no a2)   */
  const void* w;                     /* fp16 weights [num_taps*N, K], K contiguous                       */
  int32_t ldw;                       /* row pitch of w in elements (0 = K)                               */
  int32_t N;
  int32_t num_taps;                  /* 1 (linear), 3 (temporal conv), 9 (3x3 conv)                      */
  int32_t tap_dx[9], tap_dy[9];      /* per-tap shift of the tile origin along X / Y                     */
  void* out;       void* out_f32;    /* fp16 output (or fp32 if out_f32 != NULL), row pitch ldo          */
  int32_t ldo;
  const float* bias; int32_t bias_z_div;   /* bias row = z / bias_z_div (0: single row)                  */
  const void* res; int32_t ldr;      /* optional fp16 residual added in the epilogue                     */
  int32_t geglu;                     /* 1: x*gelu(gate) epilogue, weights pre-interleaved per N tile     */
  /* LayerNorm folded into the epilogue (BasicTransformerBlock norm1/2/3 -> to_q/k/v, ff.net[0]; attention.py:283-292):
   * A holds the RAW rows, w is pre-scaled by the LayerNorm weight, bias holds (W.beta + linear bias);
   * out[r,n] = rstd[r] * (acc[r,n] - mean[r] * ln_colsum[n]) + bias[n].  NULL = plain GEMM.  num_taps must be 1. */
  const float* ln_stats;             /* [rows][2] fp32 (mean, rstd) from vc_layernorm_stats                */
  const float* ln_colsum;            /* [N] fp32: sum_k w[n,k] of the fp16 weights                         */
  /* optional by-product for the NEXT LayerNorm: partial (sum, sumsq) of the fp16-rounded output, per row and 32-column chunk,
   * ln_part[(n/32) * M + row][2]; plain fp16 [M,N] outputs with N % 32 == 0 only.  vc_layernorm_stats_from_parts finishes them. */
  float* ln_part;
  /* optional output pitches in elements along Y and Z (0 = dense: ldo*X and ldo*X*Y); non-dense outputs require an fp16 output
   * with N % 32 == 0 and no residual.  Upsample (F.interpolate nearest x2, openaimodel3d.py:80-106) + 3x3 conv runs as four
   * parity sub-convolutions with 2x2 pre-summed taps on the SMALL image, each writing every second pixel of the large one. */
  int64_t ldo_y, ldo_z;
  /* optional by-product for the NEXT GroupNorm (basics.py:76-87, openaimodel3d.py:256-265): partial (sum, sumsq) of the fp16-rounded
   * output per 32-row block rb = m_tile * 4 + quadrant (m-tiles in x, y, z order, count padded to an even number), 32-column chunk and
   * piece: gn_part[((rb * (N/32) + chunk) * 4 + piece) * 2]; a chunk is cut into 4 pieces at multiples of gn_sub (10 or 8) channels.
   * vc_groupnorm_from_parts consumes them.  fp16 outputs with N % 32 == 0 and N % gn_sub == 0 only. */
  float* gn_part; int32_t gn_sub;
  /* optional: multi-GPU layout switch fused into the epilogue (see vc_gemm_peer below); NULL = write `out` locally */
  const struct vc_gemm_peer* peer;
} vc_gemm_desc;
/* Output rows of the GEMM are stored tile by tile (TMA stores through the NVLink peer mapping) into the receive buffers of the ranks
 * that own them in the OTHER layout of the frame-sharded U-Net (SURVEY.md 8e; new functionality): mode 1 = this rank's rows are
 * [(b, t_local, hw), N] and go to [(b, t, hw_local), N] on rank hw / (HW / world); mode 2 the reverse.  `out` is not written.
 * Complete the switch with vc_peer_finish_scatter (rendezvous + GroupNorm sums).  2..4 ranks, fp16 output with N % 32 == 0. */
typedef struct vc_gemm_peer {
  int32_t mode, world, rank, B, T, HW;
  int32_t f0[9];          /* rank q owns frames [f0[q], f0[q+1]) */
  void* dst[8];           /* rank q's receive buffer of the destination layout as mapped into this process */
} vc_gemm_peer;
int vc_gemm_tap(const vc_gemm_desc* d, void* stream);
/* N-tile width the kernel will use for (N, geglu): needed to interleave GEGLU weights on the host */
int vc_gemm_tile_n(int32_t N, int32_t geglu);

/* ---- fused attention, head_dim 64 ---------------------------------------------------------------------------
 * replaces: CrossAttention.forward / efficient_forward, lvdm/modules/attention.py:81-144 / 146-209
 *           (einsum-softmax-einsum or xformers.ops.memory_efficient_attention)
 */
typedef struct vc_attn_desc {
  const void* q; int32_t ldq;        /* [B, Nq, heads, 64] fp16, row pitch ldq                           */
  const void* k; int32_t ldk;        /* [Bk, Nk, heads, 64]                                              */
  const void* v; int32_t ldv;
  void* out;     int32_t ldo;        /* [B, Nq, heads*64]                                                */
  int32_t B, heads, Nq, Nk;
  int64_t kv_batch_stride;           /* elements between K/V batches; 0 = one K/V shared by all B        */
  float scale;                       /* dim_head^-0.5                                                     */
  int32_t accumulate;                /* out += result (image branch, attention.py:128-142)               */
} vc_attn_desc;
int vc_flash_attn_d64(const vc_attn_desc* d, void* stream);

/* temporal self-attention over T <= 32 frames per spatial site (TemporalTransformer, attention.py:365-412;
 * always the naive path in the reference, attention.py:66).  q/k/v rows at (t*sites + site), pitch ld. */
int vc_temporal_attn(const void* q, const void* k, const void* v, int32_t ld, void* out, int32_t ldo, int32_t T,
                     int64_t sites, int32_t heads, float scale, void* stream);

/* ---- normalisation --------------------------------------------------------------------------------------------
 * GroupNorm(32)+optional SiLU on channels-last fp16; x = concat(x1[C1], x2[C2]) along channels (x2 may be NULL).
 * replaces: GroupNormSpecific lvdm/basics.py:76-87, nn.GroupNorm in attention.py:265,331, openaimodel3d.py:256-265
 *           (5-D statistics: pass samples = B, rows_per_sample = T*H*W), ae_modules.py:15-16; SiLU openaimodel3d.py:152
 */
size_t vc_groupnorm_ws_bytes(int32_t samples);
int vc_groupnorm_nhwc(const void* x1, int32_t C1, const void* x2, int32_t C2, int32_t samples, int64_t rows_per_sample,
                      const float* gamma, const float* beta, float eps, int32_t silu, void* out, void* ws, size_t ws_bytes,
                      void* stream);
/* Split form for GroupNorm statistics that span several GPUs (site-sharded 5-D GroupNorm of the temporal blocks):
 * pass 1 writes (sum, sumsq) per group to stats[samples][32][2]; the caller all-reduces that buffer (NCCL); pass 2
 * normalises with the global row count stat_rows. */
int vc_groupnorm_stats(const void* x1, int32_t C1, const void* x2, int32_t C2, int32_t samples, int64_t rows_per_sample, float* stats,
                       void* ws, size_t ws_bytes, void* stream);
int vc_groupnorm_apply(const void* x1, int32_t C1, const void* x2, int32_t C2, int32_t samples, int64_t rows_per_sample,
                       const float* stats, int64_t stat_rows, const float* gamma, const float* beta, float eps, int32_t silu, void* out,
                       void* stream);
/* pass 2 with UN-reduced statistics: parts = [samples][n_parts][32][2] partial (sum, sumsq), summed in index order */
int vc_groupnorm_apply_parts(const void* x1, int32_t C1, int32_t samples, int64_t rows_per_sample, const float* parts, int32_t n_parts,
                             int64_t stat_rows, const float* gamma, const float* beta, float eps, int32_t silu, void* out, void* stream);
/* GroupNorm(32) (+SiLU) of concat(x1, x2) whose statistics come from the gn_part records the producing vc_gemm_tap calls left
 * (one descriptor per source): the activation is read once and written once, there is no statistics pass.
 * Sample s of the consumer covers the 32-row blocks [base, base + rb_per_sample) of the producer with
 * base = (s / samples_per_z) * rb_per_z + (s % samples_per_z) * rb_per_sample.  Every group boundary of the consumer must be a
 * multiple of `sub` channels inside each source.  ws: vc_groupnorm_parts_ws_bytes(samples) bytes. */
typedef struct vc_gn_part_geom {
  const float* part; int32_t n_chunks; int32_t sub; int64_t rb_per_z; int32_t samples_per_z; int64_t rb_per_sample;
} vc_gn_part_geom;
size_t vc_groupnorm_parts_ws_bytes(int32_t samples);
int vc_groupnorm_from_parts(const void* x1, int32_t C1, const vc_gn_part_geom* g1, const void* x2, int32_t C2, const vc_gn_part_geom* g2,
                            int32_t samples, int64_t rows_per_sample, const float* gamma, const float* beta, float eps, int32_t silu,
                            void* out, void* ws, size_t ws_bytes, void* stream);
/* statistics half of nn.LayerNorm: stats[row] = (mean, 1/sqrt(var + eps)) in fp32; the normalisation is applied by the
 * consuming vc_gemm_tap (ln_stats / ln_colsum), so the normalised activation is never written to memory */
int vc_layernorm_stats(const void* x, int64_t rows, int32_t C, float eps, float* stats, void* stream);
/* the same statistics from the partial sums a producing vc_gemm_tap left in ln_part ([C/32][rows][2] fp32): no re-read of x */
int vc_layernorm_stats_from_parts(const float* parts, int64_t rows, int32_t C, float eps, float* stats, void* stream);
/* nn.LayerNorm over the last dim (attention.py:233-235), fp16 in/out, fp32 statistics */
int vc_layernorm(const void* x, int64_t rows, int32_t C, const float* gamma, const float* beta, float eps, void* out,
                 void* stream);

/* row softmax of fp32 scores (pre-scaled by `scale`) to fp16 probabilities: the VAE AttnBlock, ae_modules.py:66-68 */
int vc_softmax_rows_f32(const float* x, int64_t rows, int64_t cols, float scale, void* out, void* stream);

/* ---- data movement ----------------------------------------------------------------------------------------------- */
int vc_upsample2x_nhwc(const void* x, void* out, int32_t N, int32_t H, int32_t W, int32_t C, void* stream); /* F.interpolate nearest x2 */
int vc_im2col3x3_s2(const void* x, void* out, int32_t N, int32_t H, int32_t W, int32_t C, int32_t pad_lo, int32_t Ho, int32_t Wo,
                    void* stream);                                                                            /* Downsample conv, openaimodel3d.py:51-77 */
int vc_ncthw_f32_to_rows_f16(const float* x, void* out, int32_t B, int32_t C, int32_t T, int64_t HW, int32_t c_off, int32_t ldo,
                             void* stream);                                                                   /* 'b c t h w -> (b t) h w c' + hybrid concat ddpm3d.py:1437-1443 */
int vc_rows_f32_to_ncthw(const float* x, int32_t ldx, float* out, int32_t B, int32_t C, int32_t T, int64_t HW, void* stream);
int vc_rows_f16_to_nchw_f32(const void* x, int32_t ldx, float* out, int32_t N, int32_t C, int64_t HW, void* stream);
int vc_cast_f32_to_f16(const float* x, void* out, int64_t n, void* stream);
int vc_add_f16(const void* a, const void* b, void* out, int64_t n, void* stream);
/* out = gelu(x), exact-erf GELU on fp16 rows (nn.GELU() between the two bias-free Linears of the Resampler FeedForward,
 * lvdm/modules/encoders/resampler.py:27-34) */
int vc_gelu_f16(const void* x, void* out, int64_t n, void* stream);

/* ---- timestep / fps embedding (fp32, tiny) -------------------------------------------------------------------------
 * replaces: timestep_embedding utils_diffusion.py:8-28; time_embed / fps_embedding / emb_layers openaimodel3d.py:370-382,164-170 */
int vc_timestep_embedding(const int64_t* t, int32_t n, int32_t dim, float* out, void* stream);
int vc_small_linear_f32(const float* x, int32_t rows, int32_t K, const float* W, const float* bias, int32_t N, int32_t silu_in,
                        float* out, const float* add, void* stream);

/* ---- fused DDIM update --------------------------------------------------------------------------------------------
 * replaces: DDIMSampler.p_sample_ddim after the two apply_model calls, lvdm/models/samplers/ddim.py:228-281,
 *           rescale_noise_cfg utils_diffusion.py:147-158, predict_{eps,start}_from_z_and_v ddpm3d.py:239-251 */
typedef struct vc_ddim_scalars {
  float cfg_scale, guidance_rescale;
  float sqrt_ac_t, sqrt_1mac_t;
  float a_prev, sigma_t;
  float scale_t, prev_scale_t;
  int32_t use_cfg;
} vc_ddim_scalars;
int vc_ddim_update(const float* x, const float* v_cond, const float* v_uncond, const float* noise, float* x_prev, float* pred_x0,
                   int64_t n, const vc_ddim_scalars* s, void* ws /* 4 * 1025 doubles */, void* stream);
/* three-way CFG of DDIMSampler (multicond): v = u + cfg_img (v_img - u) + cfg_scale (v_cond - v_img), then the same rescale / update
 * replaces: lvdm/models/samplers/ddim_multiplecond.py:227-236 (+ the shared tail :238-287) */
int vc_ddim_update3(const float* x, const float* v_cond, const float* v_uncond, const float* v_uncond_img, float cfg_img,
                    const float* noise, float* x_prev, float* pred_x0, int64_t n, const vc_ddim_scalars* s, void* ws /* 4 * 1025 doubles */, void* stream);

/* ---- multi-GPU: frame <-> site layout exchange over NVLink peer memory ------------------------------------------------
 * New functionality (the reference is single-GPU, SURVEY.md 8e).  The frame-sharded U-Net runs its spatial ops on
 * [(b, t_local, hw), C] rows and its temporal ops (TemporalTransformer attention.py:365-412, TemporalConvBlock
 * openaimodel3d.py:239-279) on [(b, t_all, hw_local), C] rows.  One kernel per switch: every rank stores its rows straight
 * into the receive buffers of the owning ranks (mapped into this process with CUDA IPC by the caller) and, for
 * frames -> sites, publishes the GroupNorm(32) partial sums of the tensor it just streamed; a device-side sequence number +
 * release/acquire flags in peer memory replace the NCCL collective.  All ranks of the group must issue the same sequence of
 * vc_peer_* calls.  After the call (in stream order) cur_stats holds [B][world][32][2] partial (sum, sumsq) of all ranks
 * (frames -> sites with with_stats, and vc_peer_groupnorm_stats): feed it to vc_groupnorm_apply_parts with n_parts = world. */
typedef struct vc_peer_comm {
  int32_t world, rank;               /* ranks of the frame group (<= 8) and this rank's index in it               */
  void* flags;                       /* own uint32[world], zero-initialised before the peers map it                 */
  void* peer_flags[8];               /* rank p's flags as mapped in this process (peer_flags[rank] == flags)        */
  void* seq;                         /* own uint32: collectives completed (zero-initialised)                        */
  void* done;                        /* own uint32: scratch (zero-initialised)                                      */
  void* stats_slots[8];              /* rank p's float[2][Bmax][world][64] as mapped here                           */
  void* cur_stats;                   /* own float[Bmax][world][64]                                                  */
  int32_t Bmax;                      /* batch samples per rank the slots were sized for (1..4)                      */
} vc_peer_comm;
int vc_enable_peer_access(int32_t peer_device);
/* IPC-shareable, zero-filled device memory (cudaMalloc) + its 64-byte cudaIpcMemHandle_t; vc_peer_open maps another process's
 * allocation with the CALLING process's current device as the accessor (lazy peer mapping), vc_peer_close / vc_peer_free undo. */
int vc_peer_alloc(size_t bytes, void** ptr, void* handle64);
int vc_peer_open(const void* handle64, void** ptr);
int vc_peer_close(void* ptr);
int vc_peer_free(void* ptr);
/* src: local fp16 rows; dst[p]: rank p's receive buffer as mapped here; f0[world+1]: frame range boundaries of the ranks.
 * to_sites = 1: [(b, t_local, hw), C] -> [(b, t_all, hw_local), C]; 0: the reverse.  ws: >= B * 512 * 64 floats. */
int vc_peer_exchange(const vc_peer_comm* c, const void* src, void* const* dst, int32_t to_sites, int32_t B, int32_t T, int32_t HW,
                     int32_t C, const int32_t* f0, int32_t with_stats, void* ws, size_t ws_bytes, void* stream);
/* GroupNorm statistics of this rank's rows + exchange with all peers -> cur_stats (the site-sharded 5-D GroupNorms in the
 * middle of a temporal block, openaimodel3d.py:256-265) */
int vc_peer_finish_scatter(const vc_peer_comm* c, const vc_gn_part_geom* geom, int32_t C, int32_t samples, void* ws, size_t ws_bytes, void* stream);
int vc_peer_groupnorm_stats(const vc_peer_comm* c, const void* x, int32_t C, int32_t samples, int64_t rows_per_sample, void* ws,
                            size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VC_B200_H */
