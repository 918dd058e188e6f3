/* pa_b200.h — C ABI of the B200-native attention-forward library (libpa_b200.so).
 *
 * Drop-in boundary for the multi-head self-attention forward that recurs in the reference
 * (changzy00/pytorch-attention, vision_transformers/):
 *     ViT.Attention.forward            ViT.py:79-89      -> pa_vit_fwd
 *     pvt.Attention.forward            pvt.py:73-91      -> pa_pvt_fwd
 *     cvt.Attention.forward            cvt.py:64-76      -> pa_cvt_fwd
 *     cswin.LePEAttention.forward      cswin.py:101-127  -> pa_cswin_lepe_fwd
 *     cswin.CSWinBlock.forward (attn)  cswin.py:176-194  -> pa_cswin_block_attn_fwd
 *     dilateformer.MultiDilatelocalAttention.forward  dilateformer.py:85-97 -> pa_dilate_fwd
 *     dilateformer.DilateBlock.forward (attn)         dilateformer.py:130   -> pa_dilate_block_attn_fwd
 *     xcit.XCA.forward                 xcit.py:245-265   -> pa_xca_fwd
 *     xcit.ClassAttention.forward      xcit.py:174-188   -> pa_class_attn_fwd
 * The reference has no FFI of its own (it is pure Python calling ATen); these entry points are what a
 * ctypes binding inside each reference module's forward would call (see INTEGRATION.md).
 *
 * Conventions
 *   - plain C structs, raw device pointers, sizes, a cudaStream_t passed as void*; no C++/torch types.
 *   - every function returns 0 on success or a negative PA_ERR_* code; pa_last_error() gives the
 *     thread-local message.  Nothing is allocated, freed or synchronised by the library: the caller
 *     owns x, parameters, y and the workspace; launches are asynchronous on the given stream.
 *   - 16-bit tensors are fp16 or bf16 (PA_DTYPE_*); biases / BN / LN / temperature vectors are fp32.
 *   - there is NO CPU fallback: on a device that is not compute capability 10.x the calls fail.
 */
#ifndef PA_B200_H
#define PA_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PA_VERSION 101

enum { PA_DTYPE_F16 = 0, PA_DTYPE_BF16 = 1, PA_DTYPE_F32 = 2 };

enum {
  PA_OK = 0,
  PA_ERR_BAD_SHAPE = -1,      /* dim % heads, head_dim unsupported, L != H*W ... (reference: AssertionError) */
  PA_ERR_UNSUPPORTED = -2,    /* dtype / mode not implemented on this path */
  PA_ERR_MISALIGNED = -3,     /* pointer or pitch not 16-byte aligned */
  PA_ERR_WORKSPACE = -4,      /* workspace missing or too small */
  PA_ERR_CUDA = -5,           /* CUDA runtime/driver error (message has the cudaError string) */
  PA_ERR_DEVICE = -6,         /* not an sm_100 device / no device */
  PA_ERR_NULL = -7            /* required pointer is NULL */
};

int pa_version(void);
const char* pa_last_error(void);
/* 0 if `device` exists and is compute capability 10.x, else PA_ERR_DEVICE. */
int pa_device_check(int device);
/* number of kernels this library has launched in the calling process (all threads). */
unsigned long long pa_launch_count(void);
/* The PA_* environment switches (experiments and fallbacks, DESIGN.md §9) are read once, at the first call into the
 * library; this re-reads them (tests and tools that flip a switch inside one process call it). */
void pa_reload_env(void);
/* debug aid: occupancy facts of the co-scheduled ViT kernel (registers, static smem, blocks per SM, resident clusters, ...) */
int pa_debug_cosched_occupancy(int dynamic_smem_bytes, int* out6);

/* ---------------------------------------------------------------- building blocks (also exported for tests) */
/* D[z][m,n] = sum_k A[z][m,k] B[z][n,k] (+bias): both operands K-major, i.e. nn.Linear / 1x1-conv layout. */
typedef struct {
  int a_dtype, b_dtype, out_dtype;   /* a,b: F16/BF16; out: F16/BF16/F32 */
  int M, N, K, Z;
  const void* A; long long lda, a_batch;   /* pitches in elements; a_batch == 0: A shared by all z */
  const void* B; long long ldb, b_batch;
  void* D;       long long ldd, d_batch;
  const float* bias;                 /* fp32, length N (bias_mode 1) or M (bias_mode 2) */
  int bias_mode;                     /* 0 none, 1 per column, 2 per row */
  int block_n;                       /* 0 = auto; else 64/96/128/192/256 */
  const void* residual;              /* optional tensor added to the result ([Z][M,N], pitch ldr), or NULL */
  long long ldr, r_batch;
  int res_dtype;                     /* F16/BF16/F32 */
  int cluster;                       /* 0 = auto; 1/2/4: CTAs per cluster sharing the B tile by TMA multicast; -2: CTA pairs (tcgen05 cta_group::2) */
} pa_gemm_args;
int pa_gemm_tn(const pa_gemm_args* a, void* stream);
/* dst[i] = (fp16 | bf16) src[i], i < n: the cast in front of a forward when the caller's activations are fp32 (the reference's
 * forward is fp32 in / fp32 out, ViT.py:79; the drop-ins' opt-in `fp32_input` mode).  Both buffers 16-byte aligned. */
int pa_cast_f32(const float* src, void* dst, long long n, int out_dtype, void* stream);
/* debug aid: CTA 0 of later GEMM launches writes per-tile clock64 stamps into this device buffer (>= 4 KiB); NULL turns it off */
void pa_debug_set_gemm_trace(void* device_buffer);

/* O[g][i, h*64+d] = sum_j softmax_j(scale * Q[g][i,h,:].K[g][j,h,:]) V[g][j,h,d];  fp16 in, fp16 out, head_dim 64,
 * any n_k
 * (blocks of keys with an online softmax beyond 256).  Q rows live in `q` with pitch ldq (elements) and group pitch q_group, head h at column q_col0+64h;
 * K and V live in one buffer `kv` at columns k_col0+64h / v_col0+64h. */
typedef struct {
  int G, H, n_q, n_k;
  const void* q;  long long ldq, q_group; int q_col0;
  const void* kv; long long ldkv, kv_group; int k_col0, v_col0;
  void* o;        long long ldo, o_group;  int o_col0;
  float scale;
  int head_dim;                      /* 0 or 64: 64-wide heads; 32: 32-wide heads */
} pa_attn_args;
int pa_attn_core(const pa_attn_args* a, void* stream);

/* ---------------------------------------------------------------- ViT.Attention  (ViT.py:67-89) */
typedef struct {
  int dtype;                 /* dtype of x and qkv_weight (F16/BF16) */
  int out_dtype;             /* dtype of y (F16/BF16/F32) */
  int B, N, C, H;            /* C % H == 0 and C / H == 64 */
  float scale;               /* head_dim ** -0.5 (ViT.py:73) */
  const void* x;             /* [B,N,C] contiguous */
  const void* qkv_weight;    /* [3C,C]  rows ordered (s,h,d), ViT.py:81 */
  const float* qkv_bias;     /* [3C] fp32 or NULL (qkv_bias=False default, ViT.py:68) */
  const void* proj_weight;   /* [C,C] fp16 */
  const float* proj_bias;    /* [C] fp32 or NULL */
  void* y;                   /* [B,N,C] */
  int topk;                  /* 0: plain softmax.  > 0: kvt.KNNAttention (kvt.py:67-94; SURVEY.md section 8 row f-4): only the topk largest
                                scores of every row take part in the softmax (kvt.py:84-87).  Needs 64-wide heads, N <= 240 and
                                topk <= N; runs as GEMM(qkv) -> per-row k-th-largest kernel -> attention core (scores below the row's
                                threshold masked) -> GEMM(proj) */
} pa_vit_args;
/* One kernel launch when N <= 256, three stream-ordered launches otherwise; all paths give bit-identical results.
 *   co-scheduled kernel (default when N <= 240, C % 64 == 0, 16-bit y): two role-specialised CTAs per SM -- the qkv / proj
 *     GEMM stream (CTA pairs, 256 TMEM columns) runs under the softmax chain of the attention stream (256 TMEM columns);
 *   sequenced kernel (otherwise): qkv GEMM -> attention -> proj GEMM phases back to back on every SM.
 * Both order their work across SMs by dependency counters kept in the workspace (zeroed by a cudaMemsetAsync on the same
 * stream) and spin-wait on them, so they need every CTA of their grid resident at once: the library launches them only on
 * a grid it has established to fit (the co-scheduled kernel: a one-off probe launch + stream synchronisation at the first
 * qualifying call per device, skipped -- together with that kernel -- while the stream is being captured).  A kernel
 * that holds SMs at the same time delays them; a wait that makes no progress for ~2 s (4e9 cycles) traps with a message
 * instead of hanging the device, which poisons the CUDA context: do not co-run them with long-lived persistent kernels.
 * Environment (read once, see pa_reload_env): PA_VIT_FUSED=0 three launches, =1 a single launch or PA_ERR_UNSUPPORTED;
 * PA_VIT_COSCHED=0 never / =1 always the co-scheduled kernel (or PA_ERR_UNSUPPORTED). */
size_t pa_vit_workspace_bytes(const pa_vit_args* a);
/* 1 = three launches, 2 = sequenced single launch, 3 = co-scheduled single launch: what the calling thread's last pa_vit_fwd did */
int pa_last_vit_path(void);
int pa_vit_fwd(const pa_vit_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- ViT.TransformerEncoder, attention half  (ViT.py:116) */
/* y = x + Attention(LayerNorm(x)): the pre-norm and the residual that surround the attention in every ViT-style block
 * (ViT.py:116, the same shape as pvt.py:106 / setr.py:88 / moat.py).  LayerNorm is this library's row kernel (fp32 statistics,
 * fp16 output = the qkv GEMM's A operand), the residual is added in the epilogue of the proj GEMM (x is read there once, no
 * separate elementwise pass, no intermediate attention output in HBM).  Launches: LayerNorm -> GEMM(qkv) -> attention core ->
 * GEMM(proj + residual). */
typedef struct {
  pa_vit_args attn;          /* attn.x = block input (dtype attn.dtype), attn.y = block output of the attention half;
                                attn.qkv_weight must be fp16 (its input is the fp16 LayerNorm output) */
  const float* ln_weight;    /* [C] layernorm1.weight */
  const float* ln_bias;      /* [C] layernorm1.bias */
  float ln_eps;
} pa_vit_block_args;
size_t pa_vit_block_attn_workspace_bytes(const pa_vit_block_args* a);
int pa_vit_block_attn_fwd(const pa_vit_block_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- bvit.Broad_Attention  (bvit.py:49-76; SURVEY.md section 8 row f-4) */
/* ViT's math with an inner width heads * dim_head that need not equal dim, no qkv bias, and q, k, v handed back to the caller
 * (BViT's parameter-free broad attention reads them from every layer, bvit.py:88-98): the qkv projection is written to a
 * caller-owned buffer instead of the workspace and forward() returns views of it.  Launches: GEMM(qkv) -> attention core ->
 * GEMM(out); without an output projection (heads == 1 and dim_head == dim: nn.Identity, bvit.py:52, 61-64) the attention core
 * writes y directly. */
typedef struct {
  int dtype, out_dtype;      /* out_dtype must be fp16 when out_weight is NULL */
  int B, N, C, H, dim_head;  /* inner = H * dim_head; dim_head a multiple of 16 from 32 to 192 */
  float scale;               /* dim_head ** -0.5 (bvit.py:55) */
  const void* x;             /* [B,N,C] */
  const void* qkv_weight;    /* [3*inner, C] (dtype): to_qkv.weight, rows ordered (q|k|v, head, d) (bvit.py:67-68) */
  const void* out_weight;    /* [C, inner] fp16: to_out.0.weight, or NULL (Identity) */
  const float* out_bias;     /* [C] or NULL */
  void* qkv;                 /* OUT [B,N,3*inner] fp16 */
  void* y;                   /* OUT [B,N,C] (Identity: [B,N,inner] with inner == C) */
} pa_bvit_args;
size_t pa_bvit_workspace_bytes(const pa_bvit_args* a);
int pa_bvit_fwd(const pa_bvit_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- pvt.Attention  (pvt.py:52-91) */
typedef struct {
  int dtype, out_dtype;
  int B, N, C, H;            /* N == Himg*Wimg, C / H == 64 */
  int Himg, Wimg, sr;        /* forward(x, H, W) and the constructor's sr_ratio */
  float scale;
  const void* x;             /* [B,N,C] */
  const void* q_weight;      /* [C,C]  (dtype) */
  const float* q_bias;       /* [C] or NULL */
  const void* kv_weight;     /* [2C,C] = cat(k.weight, v.weight); fp16 when sr > 1 (its input is the fp16 reduced map), else dtype */
  const float* kv_bias;      /* [2C] or NULL */
  const void* proj_weight;   /* [C,C] fp16 */
  const float* proj_bias;    /* [C] or NULL */
  const float* sr_weight_t;  /* [sr*sr, C] fp32: sr.0.weight [C,1,sr,sr] transposed (sr > 1) */
  const float* sr_scale;     /* [C] sr.1.weight * rsqrt(running_var + eps)  (eval BatchNorm folded) */
  const float* sr_shift;     /* [C] (sr.0.bias - running_mean) * sr_scale + sr.1.bias */
  void* y;                   /* [B,N,C] */
  /* ---- siblings of the same path (SURVEY.md section 8 row f-2); all zero / NULL = plain pvt.Attention */
  int sr_mode;               /* 0: depthwise conv + eval BatchNorm (pvt.py:67-71, cmt.py:87-91)
                                1: dense conv k = stride = sr with bias, no norm (segformer.py:27, 38-39), run as a GEMM over
                                   the non-overlapping sr x sr patches */
  const void* sr_dense_weight; /* sr_mode 1: [C, sr*sr*C] (dtype), sr.weight [C,C,sr,sr] permuted to (co, u, v, ci) */
  const float* sr_dense_bias;  /* sr_mode 1: [C] or NULL */
  const float* rel_pos;      /* cmt.Attention.forward(x, H, W, relative_pos), cmt.py:100: fp32 [H, N, M] added to
                                q k^T * scale before the softmax (M = key tokens after the reduction), or NULL.
                                Needs 64-wide heads and M <= 240 */
  const void* kv_tokens;     /* NULL, or fp16 [B, kv_count, C]: keys / values are projected from THESE tokens instead of from x
                                (sr must be 1; kv_weight fp16) -- the pooled pyramid of p2t.PoolingAttention, see pa_p2t_fwd */
  int kv_count;
} pa_pvt_args;
size_t pa_pvt_workspace_bytes(const pa_pvt_args* a);
int pa_pvt_fwd(const pa_pvt_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- pvt.Block / segformer.Block / cmt.Block, attention half */
/* y = x + Attention(LayerNorm(x), H, W [, relative_pos])   (pvt.py:106, segformer.py:76, cmt.py:131): this library's LayerNorm
 * row kernel (fp32 statistics, fp16 output) in front, the residual x added in the epilogue of the proj GEMM.  attn.q_weight
 * and (sr == 1) attn.kv_weight must be fp16: their input is the fp16 LayerNorm output. */
typedef struct {
  pa_pvt_args attn;          /* attn.x = block input, attn.y = x + attention */
  const float* ln_weight;    /* [C] norm1.weight */
  const float* ln_bias;      /* [C] norm1.bias */
  float ln_eps;
} pa_pvt_block_args;
size_t pa_pvt_block_attn_workspace_bytes(const pa_pvt_block_args* a);
int pa_pvt_block_attn_fwd(const pa_pvt_block_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- p2t.PoolingAttention  (p2t.py:46-94; SURVEY.md section 8 row f-4) */
/* Keys / values come from a pooling pyramid of the token map (p2t.py:78-86): per level l
 *     pool_l = adaptive_avg_pool2d(x as [B,C,H,W], (pool_h[l], pool_w[l]));  pool_l += d_convs[l](pool_l)   (depthwise 3x3, zero pad)
 * the levels concatenated along the token axis, LayerNorm over the channels, then kv = Linear(C, 2C).  Two small kernels build
 * those tokens (adaptive average straight from the token-major x; depthwise conv + skip + LayerNorm, one warp per pooled token),
 * the rest is the PVT path with `kv_tokens`: GEMM(q) -> GEMM(kv) -> attention core -> GEMM(proj). */
typedef struct {
  pa_pvt_args attn;          /* B, N = Himg*Wimg, C, H, scale, x, q_weight / q_bias, kv_weight (fp16 [2C,C] = kv.0.weight) / kv_bias,
                                proj_*, y; sr = 1, sr_mode = 0, kv_tokens / kv_count are filled in by the library */
  int n_levels;              /* 1..4 */
  int pool_h[4], pool_w[4];  /* round(H / pool_ratio), round(W / pool_ratio) per level (p2t.py:80) */
  const float* dconv_weight_t[4];   /* per level [9, C] fp32: d_convs[l].weight [C,1,3,3] transposed */
  const float* dconv_bias[4];       /* per level [C] fp32 or NULL */
  const float* norm_weight;  /* [C] self.norm (p2t.py:74) */
  const float* norm_bias;
  float norm_eps;
} pa_p2t_args;
size_t pa_p2t_workspace_bytes(const pa_p2t_args* a);
int pa_p2t_fwd(const pa_p2t_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- cvt.Attention  (cvt.py:48-76), NCHW in and out */
typedef struct {
  int dtype, out_dtype;
  int B, C, H, Himg, Wimg, ks;
  float scale;
  const void* x;             /* [B,C,Himg,Wimg] */
  const float* dw_weight;    /* [C, ks*ks] fp32  (conv_proj_qkv.0.weight) */
  const float* dw_scale;     /* [C] BN scale folded */
  const float* dw_shift;     /* [C] (conv bias - mean) * scale + beta */
  const void* qkv_weight;    /* [3C,C] fp16 (conv_proj_qkv.2.weight, 1x1) */
  const float* qkv_bias;     /* [3C] */
  const void* proj_weight;   /* [C,C] fp16 (proj.weight, 1x1) */
  const float* proj_bias;    /* [C] */
  void* y;                   /* [B,C,Himg,Wimg] */
  const void* residual;      /* NULL, or an NCHW tensor (dtype) added to the projection's result in its epilogue.  With ks = 1,
                                a unit depthwise tap, H = 1, scale = 1 and proj_weight = alpha * I this entry point is
                                dual_attention.PAM (attention_mechanisms/dual_attention.py:12-28): out = alpha * attn(x) + x */
} pa_cvt_args;
size_t pa_cvt_workspace_bytes(const pa_cvt_args* a);
int pa_cvt_fwd(const pa_cvt_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- xcit.XCA (xcit.py:233-265) and xcit.ClassAttention (xcit.py:159-188) */
typedef struct {
  int dtype, out_dtype;
  int B, N, C, H;            /* C / H == 64 or 32 (xcit_nano_12_p16: dim 128, 4 heads) */
  float scale;               /* ClassAttention only (XCA has no head_dim scale, xcit.py:258) */
  const void* x;             /* [B,N,C] */
  const void* qkv_weight;    /* [3C,C] (dtype) */
  const float* qkv_bias;     /* [3C] or NULL */
  const void* proj_weight;   /* [C,C] fp16 */
  const float* proj_bias;    /* [C] or NULL */
  const float* temperature;  /* [H] fp32 (XCA only) */
  void* y;                   /* [B,N,C] */
} pa_xcit_args;
size_t pa_xca_workspace_bytes(const pa_xcit_args* a);
int pa_xca_fwd(const pa_xcit_args* a, void* workspace, size_t workspace_bytes, void* stream);
/* xcit.XCABlock, attention half (xcit.py:291):  y = x + gamma1 * XCA(LayerNorm(x)).  LayerScale is folded by the caller:
 * attn.proj_weight = gamma1[:,None] * proj.weight (fp16), attn.proj_bias = gamma1 * proj.bias -- algebraically the same
 * x + O (gamma1 * Wp)^T + gamma1 * b, so the residual epilogue of the proj GEMM finishes the block.  attn.qkv_weight must be
 * fp16 (its input is the fp16 LayerNorm output).  Launches: LayerNorm -> GEMM(qkv) -> XCA core -> GEMM(proj + residual). */
typedef struct {
  pa_xcit_args attn;         /* attn.x = block input, attn.y = block output of the attention half */
  const float* ln_weight;    /* [C] norm1.weight */
  const float* ln_bias;      /* [C] norm1.bias */
  float ln_eps;
} pa_xca_block_args;
size_t pa_xca_block_attn_workspace_bytes(const pa_xca_block_args* a);
int pa_xca_block_attn_fwd(const pa_xca_block_args* a, void* workspace, size_t workspace_bytes, void* stream);
size_t pa_class_attn_workspace_bytes(const pa_xcit_args* a);
int pa_class_attn_fwd(const pa_xcit_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- cswin.LePEAttention (cswin.py:51-127) */
typedef struct {
  int B, L, C, H;            /* C = channels of this branch, C / H in {32, 64}; L == resolution^2 */
  int resolution, idx, split_size;   /* idx: -1 full window, 0 full-height stripes, 1 full-width stripes (cswin.py:62-67) */
  float scale;
  const void* q; const void* k; const void* v;   /* fp16, each [B, L, C] with row pitch ld and image pitch batch_stride */
  long long ld, batch_stride;
  const float* get_v_weight_t;   /* [9, C] fp32: get_v.weight [C,1,3,3] transposed */
  const float* get_v_bias;       /* [C] */
  void* out; long long ldo, out_batch_stride;    /* fp16 [B, L, C] */
} pa_cswin_lepe_args;
int pa_cswin_lepe_fwd(const pa_cswin_lepe_args* a, void* stream);

/* ---------------------------------------------------------------- cswin.CSWinBlock attention half (cswin.py:176-194) */
typedef struct {
  int dtype, out_dtype;
  int B, L, C, H;            /* H = num_heads of the block */
  int reso, split_size, last_stage;
  int residual;              /* 1: y = x + proj(...) (cswin.py:194); 0: y = proj(...) */
  float scale, ln_eps;
  const void* x;             /* [B,L,C] */
  const float* norm1_weight; const float* norm1_bias;
  const void* qkv_weight;    /* [3C,C] fp16 */
  const float* qkv_bias;     /* [3C] or NULL */
  const void* proj_weight;   /* [C,C] fp16 */
  const float* proj_bias;
  const float* get_v_weight_t[2];   /* per branch: [9, C/branches] fp32 */
  const float* get_v_bias[2];
  void* y;                   /* [B,L,C] */
} pa_cswin_block_args;
size_t pa_cswin_block_attn_workspace_bytes(const pa_cswin_block_args* a);
int pa_cswin_block_attn_fwd(const pa_cswin_block_args* a, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------- dilateformer.MultiDilatelocalAttention (dilateformer.py:41-97) */
/* Multi-scale dilated attention on a channels-last image x[B, Himg, Wimg, C].  qkv = 1x1 conv (a token-major GEMM), column
 * s*C + g*Cg + h*hd + d = (q/k/v, dilation group g, head h of the group, channel d), Cg = C / n_dilation.  Query (y, x) of group g
 * attends to the kernel_size^2 keys at (y + i*dilation[g] - p, x + j*dilation[g] - p), p = dilation[g]*(kernel_size-1)/2
 * (nn.Unfold, zero padding: a key outside the map has logit 0 and value 0 and still takes part in the softmax); the result of
 * head h of group g lands at column g*Cg + h*hd + d, and y = proj(O) + proj_bias.  head_dim = C / H a multiple of 8 up to 64,
 * odd kernel_size <= 7 (an even one is PA_ERR_BAD_SHAPE), 1 to 8 groups, H % n_dilation == 0, any dilation >= 1 (one beyond the
 * map is all padding but the centre tap).  Width bound: a CTA stages whole image rows of its group, so for every group
 * 4 * Wimg * pitch * min(Himg, 1 + dilation*(kernel_size-1), kernel_size) bytes must fit 227 KB, pitch = Cg rounded up to an
 * odd multiple of 8; at kernel_size 3 that is Wimg <= 807 for Cg 24, 484 for Cg 32, 345 for Cg 48.  Wider maps:
 * PA_ERR_UNSUPPORTED.
 * Launches: GEMM(qkv) -> dilated-attention kernel -> GEMM(proj).
 * The reference writes the pre-projection attention output into the caller's x (dilateformer.py:90-93 assign through a view of a
 * contiguous x); this library reads x only. */
typedef struct {
  int dtype, out_dtype;      /* x and qkv_weight: F16/BF16; y: F16/BF16/F32 */
  int B, Himg, Wimg, C, H;   /* H = num_heads */
  int kernel_size, n_dilation;
  int dilation[8];           /* dilation[g], g < n_dilation */
  float scale;               /* qk_scale or head_dim ** -0.5 (dilateformer.py:75) */
  const void* x;             /* [B,Himg,Wimg,C] */
  const void* qkv_weight;    /* [3C,C] (dtype): qkv.weight [3C,C,1,1] */
  const float* qkv_bias;     /* [3C] or NULL */
  const void* proj_weight;   /* [C,C] fp16 */
  const float* proj_bias;    /* [C] or NULL */
  void* y;                   /* [B,Himg,Wimg,C] */
} pa_dilate_args;
size_t pa_dilate_workspace_bytes(const pa_dilate_args* a);
int pa_dilate_fwd(const pa_dilate_args* a, void* workspace, size_t workspace_bytes, void* stream);
/* The dilated-attention kernel alone: o[B*Himg*Wimg, C] from a caller's qkv[B*Himg*Wimg, 3C] (both fp16, 16-byte aligned, laid out
 * as above).  Uses B, Himg, Wimg, C, H, kernel_size, n_dilation, dilation and scale of `a`. */
int pa_dilate_core(const pa_dilate_args* a, const void* qkv, void* o, void* stream);

/* ---------------------------------------------------------------- dilateformer.DilateBlock, attention half (dilateformer.py:126-130) */
/* y = x + MultiDilatelocalAttention(LayerNorm(x)) on channels-last x: this library's LayerNorm row kernel (fp32 statistics, fp16
 * output) in front, the residual x added in the epilogue of the proj GEMM.  attn.qkv_weight must be fp16 (its input is the fp16
 * LayerNorm output).  Launches: LayerNorm -> GEMM(qkv) -> dilated-attention kernel -> GEMM(proj + residual). */
typedef struct {
  pa_dilate_args attn;       /* attn.x = block input (channels-last), attn.y = block output of the attention half */
  const float* ln_weight;    /* [C] norm1.weight */
  const float* ln_bias;      /* [C] norm1.bias */
  float ln_eps;
} pa_dilate_block_args;
size_t pa_dilate_block_attn_workspace_bytes(const pa_dilate_block_args* a);
int pa_dilate_block_attn_fwd(const pa_dilate_block_args* a, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* PA_B200_H */
