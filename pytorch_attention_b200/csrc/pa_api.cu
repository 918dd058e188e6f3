// pa_api.cu — C-ABI entry points of libpa_b200.so (see include/pa_b200.h).
#include "pa_attn.cuh"
#include "pa_attn_wide.cuh"
#include "pa_gemm.cuh"
#include "pa_fused.cuh"
#include "pa_cosched.cuh"
#include "pa_host.cuh"
#include "pa_misc.cuh"
#include "pa_xca.cuh"
#include "pa_attn_win.cuh"
#include "pa_attn_proj.cuh"
#include "pa_dilate.cuh"

#include <math.h>
#include <stdlib.h>

using namespace pa;

namespace {

inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// bump allocator over the caller's workspace
struct Arena {
  uint8_t* base;
  size_t off;
  explicit Arena(void* ws) : base(reinterpret_cast<uint8_t*>(align_up(reinterpret_cast<size_t>(ws), 1024))), off(0) {}
  void* take(size_t bytes) {
    void* p = base + off;
    off += align_up(bytes, 1024);
    return p;
  }
};


// ------------------------------------------------------------------------------------------------ environment switches
// Read ONCE (first call, or pa_reload_env()): no getenv on the per-forward path.  All of them are experiments / fallbacks;
// none changes results (DESIGN.md §9).
struct EnvCfg {
  int gemm_maxworkers = 0, gemm_cluster = 0, gemm_bn = 0, gemm_balanced = 0, gemm_debug = 0, gemm_direct_store = 0;
  int attn_debug = 0, attn_direct_store = 0;
  int vit_fused = -1;        // -1 unset, 0 three launches, 1 single launch required
  int vit_cosched = -1;      // -1 unset (co-scheduled kernel when it qualifies), 0 never, 1 required
  int fused_bn1 = 0, fused_bn2 = 0;
  int cs_debug = 0, cs_lag = 0, gemm_one_set = 0, attn_two_slot = 0, cswin_two_kernels = 0;
  int cs_qtail = -1;         // the same for the last m-groups of the qkv phase
  int cs_tail = -1;          // co-scheduled kernel: m-groups at the end of the proj phase issued as 256 x 64 quarters (-1: default)
  int pvt_fused = 0;         // 1: attention core + proj GEMM as ONE kernel (pa_attn_proj.cuh; measured slower, see there)
};
std::atomic<const EnvCfg*> g_env{nullptr};
std::mutex g_env_mu;

int env_int(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}
const EnvCfg* env_load() {
  EnvCfg* c = new EnvCfg;       // a reload leaks the previous (tiny) block on purpose: concurrent readers may still hold it
  c->gemm_maxworkers = env_int("PA_GEMM_MAXWORKERS", 0);
  c->gemm_cluster = env_int("PA_GEMM_CLUSTER", 0);
  c->gemm_bn = env_int("PA_GEMM_BN", 0);
  c->gemm_balanced = getenv("PA_GEMM_BALANCED") != nullptr;
  c->gemm_debug = env_int("PA_GEMM_DEBUG", 0);
  c->gemm_direct_store = getenv("PA_GEMM_DIRECT_STORE") != nullptr;
  c->attn_debug = env_int("PA_ATTN_DEBUG", 0);
  c->attn_direct_store = getenv("PA_ATTN_DIRECT_STORE") != nullptr;
  c->vit_fused = env_int("PA_VIT_FUSED", -1);
  c->vit_cosched = env_int("PA_VIT_COSCHED", -1);
  c->fused_bn1 = env_int("PA_FUSED_BN1", 0);
  c->fused_bn2 = env_int("PA_FUSED_BN2", 0);
  c->cs_debug = env_int("PA_CS_DEBUG", 0);
  c->cs_lag = env_int("PA_CS_LAG", 0);
  c->gemm_one_set = getenv("PA_GEMM_ONE_SET") != nullptr;
  c->attn_two_slot = getenv("PA_ATTN_TWO_SLOT") != nullptr;
  c->cswin_two_kernels = getenv("PA_CSWIN_TWO_KERNELS") != nullptr;
  c->pvt_fused = env_int("PA_PVT_FUSED", 0);
  c->cs_tail = env_int("PA_CS_TAIL", -1);
  c->cs_qtail = env_int("PA_CS_QTAIL", -1);
  return c;
}
inline const EnvCfg& env() {
  const EnvCfg* c = g_env.load(std::memory_order_acquire);
  if (c) return *c;
  std::lock_guard<std::mutex> lk(g_env_mu);
  c = g_env.load(std::memory_order_acquire);
  if (!c) { c = env_load(); g_env.store(c, std::memory_order_release); }
  return *c;
}

// per-device "attribute already set" bookkeeping shared by the launchers (several host threads may drive several GPUs)
struct SmemAttr {
  std::mutex mu;
  int set[64] = {0};
  template <typename K>
  int ensure(K kernel, int bytes) {
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    std::lock_guard<std::mutex> lk(mu);
    if (set[dev] < bytes) {
      PA_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
      set[dev] = bytes;
    }
    return PA_OK;
  }
};

// ------------------------------------------------------------------------------------------------ GEMM
template <int BN, int ST, int CL, bool PAIR = false, int ESETS = 1>
int launch_gemm_cfg(const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD, GemmParams p, cudaStream_t st) {
  using Cfg = GemmCfg<BN, ST, PAIR>;
  static SmemAttr smem_attr;
  { const int rc = smem_attr.ensure(gemm_tn_kernel<BN, ST, CL, PAIR, ESETS>, Cfg::SMEM_BYTES); if (rc) return rc; }
  p.m_groups = (p.m_tiles + CL - 1) / CL;
  if (!(PAIR && BN == 256)) p.balanced = 0;
  const int supertiles = p.m_groups * p.n_tiles * p.Z;
  int max_clusters = num_sms() / CL;
  if (const int v = env().gemm_maxworkers) {   // experiment: contention vs number of active workers
    if (v > 0 && v < max_clusters) max_clusters = v;
  }
  const int nclusters = supertiles < max_clusters ? supertiles : max_clusters;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(nclusters * CL);
  cfg.blockDim = dim3(128 + 128 * ESETS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CL;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = CL > 1 ? 1 : 0;
  PA_CUDA_OK(cudaLaunchKernelEx(&cfg, gemm_tn_kernel<BN, ST, CL, PAIR, ESETS>, tmA, tmB, tmD, p));
  launch_counter()++;
  return PA_OK;
}

template <int BN, int ST>
int launch_gemm_cl(int cl, const CUtensorMap& tmA, const CUtensorMap& tmB, const CUtensorMap& tmD, const GemmParams& p,
                   cudaStream_t st) {
  if (cl == -2) {
    constexpr int PST = (ST * (128 + BN) * 128) / ((128 + BN / 2) * 128) < 8 ? (ST * (128 + BN)) / (128 + BN / 2) : 8;
    // two epilogue warp sets whenever the staged-store path is taken and the tile is wide enough for the drain to matter
    if (BN >= 128 && p.tma_store && !env().gemm_one_set) return launch_gemm_cfg<BN, PST, 2, true, 2>(tmA, tmB, tmD, p, st);
    return launch_gemm_cfg<BN, PST, 2, true>(tmA, tmB, tmD, p, st);
  }
  if (cl == 4) return launch_gemm_cfg<BN, ST, 4>(tmA, tmB, tmD, p, st);
  if (cl == 2) return launch_gemm_cfg<BN, ST, 2>(tmA, tmB, tmD, p, st);
  return launch_gemm_cfg<BN, ST, 1>(tmA, tmB, tmD, p, st);
}

long long* g_gemm_trace = nullptr;   // debug hook, see pa_debug_set_gemm_trace
thread_local int t_last_vit_path = 0; // which path the calling thread's last pa_vit_fwd took (see pa_last_vit_path)

int pick_cluster(int m_tiles) {
  const int v = env().gemm_cluster;
  if (v == 1 || v == 2 || v == 4 || v == -2) return v;
  return m_tiles >= 2 ? -2 : 1;
}

int pick_block_n(int M, int N, int K, int Z, bool pair) {
  {
    const int v = env().gemm_bn;
    if (v == 64 || v == 96 || v == 128 || v == 192 || v == 256) return v;
  }
  const int cands[5] = {256, 192, 128, 96, 64};
  // workers: CTA pairs working on 256-row tiles, or single CTAs on 128-row tiles
  const int workers = pair ? num_sms() / 2 : num_sms();
  const int m_tiles = pair ? (M + 255) / 256 : (M + 127) / 128;
  const int num_kb = (K + 63) / 64;
  double best = 1e30;
  int best_bn = 128;
  for (int i = 0; i < 5; ++i) {
    const int bn = cands[i];
    const long long tiles = (long long)m_tiles * ((N + bn - 1) / bn) * Z;
    const long long waves = (tiles + workers - 1) / workers;
    // MMA cycles per tile (the tensor core walks N in 64-column steps of 32 cycles) + fixed per-tile overhead;
    // narrow tiles pay more shared-memory traffic per flop
    // Pair tiles narrower than 256 columns are bound by the shared-memory port, not by the tensor pipe: per k-block a CTA writes
    // and reads (128 + bn/2) rows of 128 B against 128 B/clk, the pipe needs 2*bn cycles -> rate cap 2*bn / (128 + bn/2)
    // (256: 1.0, 192: 0.86, 128: 0.67).  Measured (tools/gemm_trace2.py): 192-wide tiles take 5.0 k cycles per mainloop instead
    // of 4.6 k, so 450 tiles of 256 beat 600 tiles of 192 on 74 pairs although 6.08 waves round up to 7.
    double per_tile = 2.0 * num_kb * bn;
    if (pair) { const double cap = 2.0 * bn / (128.0 + bn / 2.0); if (cap < 1.0) per_tile /= cap; }
    else if (bn < 128) per_tile *= 1.0 + 0.10 * (128.0 / bn - 1.0);
    per_tile += 700.0;
    const double cost = waves * per_tile + 0.5 * per_tile;     // + the exposed epilogue of the last tile
    if (cost < best * 0.999) { best = cost; best_bn = bn; }
  }
  return best_bn;
}

struct GemmPlan {
  CUtensorMap tmA, tmB, tmD;
  GemmParams p;
  int bn, cl;
};

// validates, picks the tile configuration (or takes force_bn / force_cl), builds tensor maps and kernel parameters
int gemm_prepare(const pa_gemm_args* a, GemmPlan* plan, int force_bn = 0, int force_cl = 0) {
  CUtensorMap& tmA = plan->tmA; CUtensorMap& tmB = plan->tmB; CUtensorMap& tmD = plan->tmD;
  GemmParams& p = plan->p;
  if (!a) return fail(PA_ERR_NULL, "pa_gemm_tn: args is NULL");
  if (!a->A || !a->B || !a->D) return fail(PA_ERR_NULL, "pa_gemm_tn: A/B/D must be non-NULL");
  if (a->M <= 0 || a->N <= 0 || a->K <= 0 || a->Z <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_gemm_tn: M,N,K,Z must be positive");
  if (a->K % 8 != 0) return fail(PA_ERR_BAD_SHAPE, "pa_gemm_tn: K=%d must be a multiple of 8", a->K);
  if (a->a_dtype > 1 || a->b_dtype > 1 || a->a_dtype < 0 || a->b_dtype < 0) return fail(PA_ERR_UNSUPPORTED, "pa_gemm_tn: operands must be fp16/bf16");
  if (a->out_dtype < 0 || a->out_dtype > 2) return fail(PA_ERR_UNSUPPORTED, "pa_gemm_tn: bad out_dtype");
  if (a->bias_mode != 0 && !a->bias) return fail(PA_ERR_NULL, "pa_gemm_tn: bias_mode set but bias is NULL");
  int rc = current_device_check();
  if (rc) return rc;

  int cl = force_cl ? force_cl : a->cluster ? a->cluster : pick_cluster((a->M + 127) / 128);
  int bn = force_bn ? force_bn : a->block_n ? a->block_n : pick_block_n(a->M, a->N, a->K, a->Z, cl == -2);
  if (!a->block_n && cl == -2 && env().gemm_balanced) bn = 256;   // experimental: balanced unit walk needs 256-wide tiles
  if (cl != 1 && cl != 2 && cl != 4 && cl != -2) return fail(PA_ERR_UNSUPPORTED, "pa_gemm_tn: cluster %d not in {1,2,4,-2}", cl);
  if (bn == 96 && cl == 4) cl = 2;          // B slices must stay whole 8-row swizzle atoms
  const bool pair = (cl == -2);             // cta_group::2: CTA pairs, 256-row tiles, each CTA stages half of B
  // balanced unit partition (32-row B boxes): measured 2 % better than the classic order at BLOCK_N 256 but worse than
  // classic BLOCK_N 192 on the ViT shapes (four small TMA boxes per k-block, less A-tile sharing in L2) -> opt-in only
  const bool balanced = pair && bn == 256 && env().gemm_balanced;
  const int b_box_rows = balanced ? 32 : pair ? bn / 2 : bn / cl;
  {
    const int za = a->a_batch ? a->Z : 1;
    uint64_t dims[3] = {(uint64_t)a->K, (uint64_t)a->M, (uint64_t)za};
    uint64_t str[2] = {(uint64_t)a->lda * 2, (uint64_t)(a->a_batch ? a->a_batch : (long long)a->lda * a->M) * 2};
    uint32_t box[3] = {64, 128, 1};
    rc = make_tmap_16b(&tmA, a->a_dtype, a->A, 3, dims, str, box);
    if (rc) return rc;
  }
  {
    const int zb = a->b_batch ? a->Z : 1;
    uint64_t dims[3] = {(uint64_t)a->K, (uint64_t)a->N, (uint64_t)zb};
    uint64_t str[2] = {(uint64_t)a->ldb * 2, (uint64_t)(a->b_batch ? a->b_batch : (long long)a->ldb * a->N) * 2};
    uint32_t box[3] = {64, (uint32_t)b_box_rows, 1};
    rc = make_tmap_16b(&tmB, a->b_dtype, a->B, 3, dims, str, box);
    if (rc) return rc;
  }
  p.M = a->M; p.N = a->N; p.K = a->K; p.Z = a->Z;
  p.m_tiles = (a->M + 127) / 128;
  p.n_tiles = (a->N + bn - 1) / bn;
  p.a_batched = a->a_batch != 0;
  p.b_batched = a->b_batch != 0;
  p.D = a->D; p.ldd = a->ldd; p.d_batch = a->d_batch;
  p.bias = a->bias; p.bias_mode = a->bias_mode; p.out_dtype = a->out_dtype;
  p.residual = a->residual; p.ldr = a->ldr; p.r_batch = a->r_batch; p.res_dtype = a->res_dtype;
  p.idesc = make_idesc(pair ? 256 : 128, bn, a->a_dtype, a->b_dtype, 0, 0);
  p.trace = g_gemm_trace;
  p.balanced = balanced ? 1 : 0;
  p.wait_ctr = nullptr; p.wait_rows = 1; p.wait_target = 0; p.signal_ctr = nullptr; p.worker_shift = 0;
  p.n_units = (a->N + 63) / 64;
  p.debug_flags = env().gemm_debug;
  // output map for the staged TMA-store epilogue (128 x 32 sub-tiles); needs 16-byte aligned base and pitches
  const int elt = a->out_dtype == PA_DTYPE_F32 ? 4 : 2;
  p.tma_store = ((reinterpret_cast<uintptr_t>(a->D) & 15) == 0) && ((a->ldd * elt) % 16 == 0) &&
                (a->Z == 1 || (a->d_batch * elt) % 16 == 0) && !env().gemm_direct_store;
  tmD = tmA;
  if (p.tma_store) {
    uint64_t dims[3] = {(uint64_t)a->N, (uint64_t)a->M, (uint64_t)a->Z};
    uint64_t str[2] = {(uint64_t)a->ldd * elt, (uint64_t)(a->Z > 1 ? a->d_batch : a->ldd * (long long)a->M) * elt};
    uint32_t box[3] = {32, 128, 1};
    rc = make_tmap_16b(&tmD, a->out_dtype, a->D, 3, dims, str, box, elt == 4 ? TM_SWZ_128 : TM_SWZ_64);
    if (rc) return rc;
  }
  plan->bn = bn; plan->cl = cl;
  return PA_OK;
}

int gemm_impl(const pa_gemm_args* a, cudaStream_t st) {
  GemmPlan plan;
  int rc = gemm_prepare(a, &plan);
  if (rc) return rc;
  const CUtensorMap& tmA = plan.tmA; const CUtensorMap& tmB = plan.tmB; const CUtensorMap& tmD = plan.tmD;
  const GemmParams& p = plan.p;
  const int bn = plan.bn, cl = plan.cl;
  switch (bn) {
    case 256: return launch_gemm_cl<256, 4>(cl, tmA, tmB, tmD, p, st);
    case 192: return launch_gemm_cl<192, 4>(cl, tmA, tmB, tmD, p, st);
    case 128: return launch_gemm_cl<128, 6>(cl, tmA, tmB, tmD, p, st);
    case 96:  return launch_gemm_cl<96, 6>(cl, tmA, tmB, tmD, p, st);
    case 64:  return launch_gemm_cl<64, 8>(cl, tmA, tmB, tmD, p, st);
    default: return fail(PA_ERR_UNSUPPORTED, "pa_gemm_tn: block_n %d not in {64,96,128,192,256}", bn);
  }
}

// small helper for the plain 2-D "y = x W^T + b" uses
int linear(const void* x, int x_dtype, long long ldx, const void* w, int w_dtype, const float* bias, void* y, int y_dtype,
           long long ldy, long long M, int N, int K, cudaStream_t st, const void* residual = nullptr, long long ldr = 0,
           int res_dtype = 0) {
  pa_gemm_args g = {};
  g.a_dtype = x_dtype; g.b_dtype = w_dtype; g.out_dtype = y_dtype;
  g.M = (int)M; g.N = N; g.K = K; g.Z = 1;
  g.A = x; g.lda = ldx; g.B = w; g.ldb = K; g.D = y; g.ldd = ldy;
  g.bias = bias; g.bias_mode = bias ? 1 : 0;
  g.residual = residual; g.ldr = ldr; g.res_dtype = res_dtype;
  return gemm_impl(&g, st);
}

// ------------------------------------------------------------------------------------------------ attention core
struct AttnLaunch {
  int hd;                 // 64 or 32
  bool windowed;
  int G, H, n_q, n_k;     // non-windowed: G groups of n_q / n_k rows.  windowed: filled from the geometry below
  const void *q, *k, *v;
  long long ldq, q_group; // row pitch / group pitch of q (elements); windowed: ldq = token pitch, q_group = image pitch
  long long ldk, k_group; // same for k and v (they share pitches)
  int q_col0, k_col0, v_col0;
  void* o; long long ldo, o_group; int o_col0;
  float scale;
  int B, R, H_sp, W_sp;   // windowed: images, resolution, window shape
  int add_into_out;
  const float* rel_pos;   // additive score bias [H, n_q, n_k] fp32 before the softmax (cmt.py:100), or nullptr
  const float* row_thresh;  // per-row threshold on the raw scores [G, H, n_q] (kvt.py:84-87), or nullptr
};

template <int HD, bool WIN>
int launch_attn_t(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const CUtensorMap& to,
                  const AttnParams& p, int smem, cudaStream_t st) {
  static SmemAttr smem_attr;
  { const int rc = smem_attr.ensure(attn_core_kernel<HD, WIN>, smem); if (rc) return rc; }
  const int grid = p.items < num_sms() ? p.items : num_sms();
  attn_core_kernel<HD, WIN><<<grid, ATTN_THREADS, smem, st>>>(tq, tk, tv, to, p);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return PA_OK;
}

struct AttnPlan {
  CUtensorMap tq, tk, tv, to;
  AttnParams p;
  int smem;
};

int attn_prepare(const AttnLaunch& a, AttnPlan* plan) {
  CUtensorMap& tq = plan->tq; CUtensorMap& tk = plan->tk; CUtensorMap& tv = plan->tv; CUtensorMap& to = plan->to;
  AttnParams& p = plan->p;
  if (a.hd != 64 && a.hd != 32) return fail(PA_ERR_UNSUPPORTED, "attention core: head_dim %d unsupported (multiples of 16 from 32 to 192)", a.hd);
  if (!(a.scale > 0.f)) return fail(PA_ERR_UNSUPPORTED, "attention core: scale must be > 0");
  if (a.ldo % 8 || a.o_col0 % 8 || a.o_group % 8 || (reinterpret_cast<uintptr_t>(a.o) & 15))
    return fail(PA_ERR_MISALIGNED, "attention core: output pitch/offset must be multiples of 8 elements");
  int rc = current_device_check();
  if (rc) return rc;
  const int hd = a.hd;
  const int kb_max_multi = 256 - hd;
  const TmapSwizzle swz = hd == 64 ? TM_SWZ_128 : TM_SWZ_64;

  p = AttnParams{};
  p.wait_ctr = nullptr; p.signal_ctr = nullptr; p.wait_target = 0; p.wait_rows_per_group = 0; p.cta_shift = 0;
  p.H = a.H;
  p.q_col0 = a.q_col0; p.k_col0 = a.k_col0; p.v_col0 = a.v_col0;
  p.O = a.o; p.ldo = a.ldo; p.o_group = a.o_group; p.o_col0 = a.o_col0;
  p.scale_log2e = a.scale * 1.4426950408889634f;
  p.add_into_out = a.add_into_out;
  p.rel_pos = a.rel_pos; p.rel_mul = 1.f / a.scale; p.row_thresh = a.row_thresh;
  p.trace = g_gemm_trace;
  p.debug_flags = env().attn_debug;
  if (!a.windowed) {
    p.G = a.G; p.n_q = a.n_q; p.n_k = a.n_k;
    if (a.n_k <= 256) { p.nkb = 1; p.kb = (a.n_k + 15) / 16 * 16; }
    else { p.kb = kb_max_multi; p.nkb = (a.n_k + p.kb - 1) / p.kb; }
    p.kb_rows = p.kb;
    {
      uint64_t dims[3] = {(uint64_t)a.ldq, (uint64_t)a.n_q, (uint64_t)a.G};
      uint64_t str[2] = {(uint64_t)a.ldq * 2, (uint64_t)a.q_group * 2};
      uint32_t box[3] = {(uint32_t)hd, 128, 1};
      if ((rc = make_tmap_16b(&tq, PA_DTYPE_F16, a.q, 3, dims, str, box, swz))) return rc;
    }
    {
      uint64_t dims[3] = {(uint64_t)a.ldk, (uint64_t)a.n_k, (uint64_t)a.G};
      uint64_t str[2] = {(uint64_t)a.ldk * 2, (uint64_t)a.k_group * 2};
      uint32_t box[3] = {(uint32_t)hd, (uint32_t)p.kb, 1};
      if ((rc = make_tmap_16b(&tk, PA_DTYPE_F16, a.k, 3, dims, str, box, swz))) return rc;
      if ((rc = make_tmap_16b(&tv, PA_DTYPE_F16, a.v, 3, dims, str, box, swz))) return rc;
    }
  } else {
    const int R = a.R, Hs = a.H_sp, Ws = a.W_sp;
    if (R % Hs || R % Ws) return fail(PA_ERR_BAD_SHAPE, "windowed attention: resolution %d not divisible by window %dx%d", R, Hs, Ws);
    const int nI = R / Hs, nJ = R / Ws, Nw = Hs * Ws;
    p.R = R; p.H_sp = Hs; p.W_sp = Ws; p.nJ = nJ; p.nWin = nI * nJ;
    p.G = a.B * p.nWin; p.n_q = Nw; p.n_k = Nw;
    if (Ws > 256) return fail(PA_ERR_UNSUPPORTED, "windowed attention: window width %d > 256", Ws);
    if (Nw <= 256) { p.h_box = Hs; p.nkb = 1; p.kb_rows = Nw; p.kb = (Nw + 15) / 16 * 16; }
    else {
      int hb = kb_max_multi / Ws;
      while (hb > 0 && (Ws * hb) % 8 != 0) --hb;       // block buffers must start on an 8-row swizzle atom
      if (hb <= 0) return fail(PA_ERR_UNSUPPORTED, "windowed attention: cannot block a %dx%d window", Hs, Ws);
      p.h_box = hb; p.kb_rows = Ws * hb; p.kb = (p.kb_rows + 15) / 16 * 16; p.nkb = (Hs + hb - 1) / hb;
    }
    if (p.nkb * p.kb_rows > 512) return fail(PA_ERR_UNSUPPORTED, "windowed attention: window of %d tokens too large", Nw);
    // 5-D view of the token matrix: {channel, col in window, window col, row in image-window, image*window row}
    auto mk = [&](CUtensorMap* t, const void* base, long long ld, long long img_pitch) -> int {
      if (img_pitch != (long long)R * R * ld) return fail(PA_ERR_UNSUPPORTED, "windowed attention: image pitch must equal L * row pitch");
      uint64_t dims[5] = {(uint64_t)ld, (uint64_t)Ws, (uint64_t)nJ, (uint64_t)Hs, (uint64_t)a.B * nI};
      uint64_t str[4] = {(uint64_t)ld * 2, (uint64_t)Ws * ld * 2, (uint64_t)R * ld * 2, (uint64_t)Hs * R * ld * 2};
      uint32_t box[5] = {(uint32_t)hd, (uint32_t)Ws, 1, (uint32_t)p.h_box, 1};
      return make_tmap_16b(t, PA_DTYPE_F16, base, 5, dims, str, box, swz);
    };
    if ((rc = mk(&tq, a.q, a.ldq, a.q_group))) return rc;
    if ((rc = mk(&tk, a.k, a.ldk, a.k_group))) return rc;
    if ((rc = mk(&tv, a.v, a.ldk, a.k_group))) return rc;
  }
  if (p.nkb > 1 && p.kb > kb_max_multi) return fail(PA_ERR_UNSUPPORTED, "attention core: key block %d too wide", p.kb);
  p.q_tiles = (p.n_q + 127) / 128;
  p.pairs = (p.q_tiles + 1) / 2;
  p.items = p.G * p.H * p.pairs;
  p.idesc_s = make_idesc(128, p.kb, PA_F16, PA_F16, 0, 0);
  p.idesc_o = make_idesc(128, hd, PA_F16, PA_F16, 0, 1);
  // staged TMA-store epilogue when the plan still fits (and rows are consecutive tokens), else direct stores
  bool staged = !a.windowed && !env().attn_direct_store &&
                attn_smem_bytes(hd, false, p.nkb, p.kb, p.kb_rows, true) <= 227 * 1024;
  const int smem = attn_smem_bytes(hd, a.windowed, p.nkb, p.kb, p.kb_rows, staged);
  if (smem > 227 * 1024) return fail(PA_ERR_UNSUPPORTED, "attention core: shared memory plan %d B too large", smem);
  // output map for the staged TMA-store epilogue (non-windowed): {columns, rows of a group, groups}, box {hd, 128, 1}
  to = tq;
  p.tma_store = 0;
  if (staged) {
    uint64_t dims[3] = {(uint64_t)a.ldo, (uint64_t)a.n_q, (uint64_t)a.G};
    uint64_t str[2] = {(uint64_t)a.ldo * 2, (uint64_t)a.o_group * 2};
    uint32_t box[3] = {(uint32_t)hd, 128, 1};
    if ((rc = make_tmap_16b(&to, PA_DTYPE_F16, a.o, 3, dims, str, box, swz))) return rc;
    p.tma_store = 1;
  }
  plan->smem = smem;
  return PA_OK;
}

// head dims 48 / 80 / 96 / ... / 192 (multiples of 16 other than 32 and 64): pa_attn_wide.cuh (panelled operands, 64-key blocks, online softmax, 2 CTAs per SM)
template <int HD>
int launch_attn_wide(const AttnLaunch& a, cudaStream_t st) {
  using Cfg = AttnWideCfg<HD>;
  int rc;
  CUtensorMap tq, tk, tv;
  const TmapSwizzle swz = Cfg::W == 64 ? TM_SWZ_128 : Cfg::W == 32 ? TM_SWZ_64 : TM_SWZ_32;
  {
    uint64_t dims[3] = {(uint64_t)a.ldq, (uint64_t)a.n_q, (uint64_t)a.G};
    uint64_t str[2] = {(uint64_t)a.ldq * 2, (uint64_t)a.q_group * 2};
    uint32_t box[3] = {(uint32_t)Cfg::W, 128, 1};
    if ((rc = make_tmap_16b(&tq, PA_DTYPE_F16, a.q, 3, dims, str, box, swz))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)a.ldk, (uint64_t)a.n_k, (uint64_t)a.G};
    uint64_t str[2] = {(uint64_t)a.ldk * 2, (uint64_t)a.k_group * 2};
    uint32_t box[3] = {(uint32_t)Cfg::W, (uint32_t)AW_KB, 1};
    if ((rc = make_tmap_16b(&tk, PA_DTYPE_F16, a.k, 3, dims, str, box, swz))) return rc;
    if ((rc = make_tmap_16b(&tv, PA_DTYPE_F16, a.v, 3, dims, str, box, swz))) return rc;
  }
  AttnWideParams p = {};
  p.G = a.G; p.H = a.H; p.n_q = a.n_q; p.n_k = a.n_k;
  p.nkb = (a.n_k + AW_KB - 1) / AW_KB;
  p.q_tiles = (a.n_q + 127) / 128;
  p.units = a.G * a.H * p.q_tiles;
  p.q_col0 = a.q_col0; p.k_col0 = a.k_col0; p.v_col0 = a.v_col0;
  p.O = a.o; p.ldo = a.ldo; p.o_group = a.o_group; p.o_col0 = a.o_col0;
  p.scale_log2e = a.scale * 1.4426950408889634f;
  p.idesc_s = make_idesc(128, AW_KB, PA_F16, PA_F16, 0, 0);
  p.idesc_o = make_idesc(128, Cfg::W, PA_F16, PA_F16, 0, 1);
  static SmemAttr smem_attr;
  if ((rc = smem_attr.ensure(attn_wide_kernel<HD>, Cfg::SMEM_BYTES))) return rc;
  const int cap = 2 * num_sms();
  const int grid = p.units < cap ? p.units : cap;
  attn_wide_kernel<HD><<<grid, AW_THREADS, Cfg::SMEM_BYTES, st>>>(tq, tk, tv, p);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return PA_OK;
}

inline bool attn_wide_hd(int hd) { return hd % 16 == 0 && hd >= 48 && hd <= 192 && hd != 64; }
inline bool attn_hd_ok(int hd) { return hd == 32 || hd == 64 || attn_wide_hd(hd); }

int launch_attn_single_slot(const AttnPlan& plan, cudaStream_t st);   // below (needs pa_cosched.cuh's kernel)

int attn_launch(const AttnLaunch& a, cudaStream_t st) {
  if (attn_wide_hd(a.hd)) {
    if (a.rel_pos || a.row_thresh) return fail(PA_ERR_UNSUPPORTED, "attention core with relative_pos / top-k: needs 64-wide heads (got %d)", a.hd);
    if (a.windowed) return fail(PA_ERR_UNSUPPORTED, "windowed attention: head_dim %d unsupported (32 or 64)", a.hd);
    if (!(a.scale > 0.f)) return fail(PA_ERR_UNSUPPORTED, "attention core: scale must be > 0");
    if (a.ldo % 8 || a.o_col0 % 8 || a.o_group % 8 || (reinterpret_cast<uintptr_t>(a.o) & 15))
      return fail(PA_ERR_MISALIGNED, "attention core: output pitch/offset must be multiples of 8 elements");
    int rc = current_device_check();
    if (rc) return rc;
    switch (a.hd) {
      case 48: return launch_attn_wide<48>(a, st);
      case 80: return launch_attn_wide<80>(a, st);
      case 96: return launch_attn_wide<96>(a, st);
      case 112: return launch_attn_wide<112>(a, st);
      case 128: return launch_attn_wide<128>(a, st);
      case 144: return launch_attn_wide<144>(a, st);
      case 160: return launch_attn_wide<160>(a, st);
      case 176: return launch_attn_wide<176>(a, st);
      default: return launch_attn_wide<192>(a, st);
    }
  }
  AttnPlan plan;
  int rc = attn_prepare(a, &plan);
  if (rc) return rc;
  const int hd = a.hd;
  if (a.rel_pos || a.row_thresh) {
    // the score bias / row threshold exist in the single-slot kernel only: 64-wide heads, at most 240 keys
    if (hd != 64 || a.windowed || plan.p.nkb != 1 || !plan.p.tma_store || plan.p.kb > 240)
      return fail(PA_ERR_UNSUPPORTED, "attention core with relative_pos / top-k: needs 64-wide heads and at most 240 keys (got head_dim %d, %d keys)", hd, a.n_k);
    return launch_attn_single_slot(plan, st);
  }
  // 64-wide heads, one key block, staged output: two single-slot CTAs per SM (pa_cosched.cuh's attention role as a kernel)
  if (hd == 64 && !a.windowed && plan.p.nkb == 1 && plan.p.tma_store && plan.p.kb <= 240 && !env().attn_two_slot)
    return launch_attn_single_slot(plan, st);
  if (hd == 64) return a.windowed ? launch_attn_t<64, true>(plan.tq, plan.tk, plan.tv, plan.to, plan.p, plan.smem, st)
                                  : launch_attn_t<64, false>(plan.tq, plan.tk, plan.tv, plan.to, plan.p, plan.smem, st);
  return a.windowed ? launch_attn_t<32, true>(plan.tq, plan.tk, plan.tv, plan.to, plan.p, plan.smem, st)
                    : launch_attn_t<32, false>(plan.tq, plan.tk, plan.tv, plan.to, plan.p, plan.smem, st);
}

template <bool RELPOS>
int launch_attn_single_slot_t(const AttnPlan& plan, cudaStream_t st) {
  CsParams cp = {};
  cp.at = plan.p;
  cp.at.wait_ctr = nullptr; cp.at.signal_ctr = nullptr;
  const int smem = cs_attn_bar_offset(plan.p.kb) + 1024;
  static SmemAttr smem_attr;
  int rc = smem_attr.ensure(attn_single_slot_kernel<RELPOS>, smem);
  if (rc) return rc;
  {
    static std::mutex mu;
    static bool carve[64];
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    if (!carve[dev & 63]) {
      PA_CUDA_OK(cudaFuncSetAttribute(attn_single_slot_kernel<RELPOS>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      carve[dev & 63] = true;
    }
  }
  const int units = plan.p.G * plan.p.H * plan.p.q_tiles;
  const int cap = 2 * num_sms();
  attn_single_slot_kernel<RELPOS><<<units < cap ? units : cap, CS_THREADS, smem, st>>>(plan.tq, plan.tk, plan.tv, plan.to, cp);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return PA_OK;
}
int launch_attn_single_slot(const AttnPlan& plan, cudaStream_t st) {
  return (plan.p.rel_pos || plan.p.row_thresh) ? launch_attn_single_slot_t<true>(plan, st) : launch_attn_single_slot_t<false>(plan, st);
}

// attention core + output projection in one kernel (pa_attn_proj.cuh): 64-wide heads, at most 64 keys, 128 <= C <= 512, 16-bit y
inline bool attn_proj_ok(const AttnLaunch& a, int C, int y_dtype) {
  return a.hd == 64 && !a.windowed && a.n_k <= 64 && C == a.H * 64 && C >= 128 && C <= 512 && y_dtype != PA_DTYPE_F32 &&
         a.rel_pos == nullptr && !a.add_into_out;
}
int launch_attn_proj(const AttnLaunch& a, const void* wp, const float* bias, void* y, int y_dtype, cudaStream_t st) {
  int rc;
  const int C = a.H * 64;
  AttnProjParams p = {};
  p.G = a.G; p.H = a.H; p.n_q = a.n_q; p.n_k = a.n_k; p.kb = (a.n_k + 15) / 16 * 16;
  p.q_tiles = (a.n_q + 127) / 128; p.units = a.G * p.q_tiles; p.C = C;
  p.q_col0 = a.q_col0; p.k_col0 = a.k_col0; p.v_col0 = a.v_col0;
  p.scale_log2e = a.scale * 1.4426950408889634f;
  p.bias = bias; p.out_dtype = y_dtype;
  p.idesc_s = make_idesc(128, p.kb, PA_F16, PA_F16, 0, 0);
  p.idesc_o = make_idesc(128, 64, PA_F16, PA_F16, 0, 1);
  p.idesc_y = make_idesc(128, 128, PA_F16, PA_F16, 0, 0);
  p.trace = g_gemm_trace;
  CUtensorMap tq, tk, tv, tw, ty;
  {
    uint64_t dims[3] = {(uint64_t)a.ldq, (uint64_t)a.n_q, (uint64_t)a.G};
    uint64_t str[2] = {(uint64_t)a.ldq * 2, (uint64_t)a.q_group * 2};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_16b(&tq, PA_DTYPE_F16, a.q, 3, dims, str, box, TM_SWZ_128))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)a.ldk, (uint64_t)a.n_k, (uint64_t)a.G};
    uint64_t str[2] = {(uint64_t)a.ldk * 2, (uint64_t)a.k_group * 2};
    uint32_t box[3] = {64, (uint32_t)p.kb, 1};
    if ((rc = make_tmap_16b(&tk, PA_DTYPE_F16, a.k, 3, dims, str, box, TM_SWZ_128))) return rc;
    if ((rc = make_tmap_16b(&tv, PA_DTYPE_F16, a.v, 3, dims, str, box, TM_SWZ_128))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)C, (uint64_t)C, 1};
    uint64_t str[2] = {(uint64_t)C * 2, (uint64_t)C * C * 2};
    uint32_t box[3] = {64, 64, 1};             // half of a [128 n x 64 k] tile: each CTA of a pair fetches one and multicasts it
    if ((rc = make_tmap_16b(&tw, PA_DTYPE_F16, wp, 3, dims, str, box, TM_SWZ_128))) return rc;
  }
  {
    uint64_t dims[3] = {(uint64_t)C, (uint64_t)a.n_q, (uint64_t)a.G};
    uint64_t str[2] = {(uint64_t)C * 2, (uint64_t)a.n_q * C * 2};
    uint32_t box[3] = {32, 32, 1};
    if ((rc = make_tmap_16b(&ty, y_dtype, y, 3, dims, str, box, TM_SWZ_64))) return rc;
  }
  static SmemAttr smem_attr;
  if ((rc = smem_attr.ensure(attn_proj_kernel, AP_SMEM_BYTES))) return rc;
  const int max_pairs = num_sms() / 2, want_pairs = (p.units + 1) / 2;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(2 * (want_pairs < max_pairs ? want_pairs : max_pairs));
  cfg.blockDim = dim3(AP_THREADS);
  cfg.dynamicSmemBytes = AP_SMEM_BYTES;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  PA_CUDA_OK(cudaLaunchKernelEx(&cfg, attn_proj_kernel, tq, tk, tv, tw, ty, p));
  launch_counter()++;
  return PA_OK;
}

int attn_impl(const pa_attn_args* a, cudaStream_t st) {
  if (!a) return fail(PA_ERR_NULL, "pa_attn_core: args is NULL");
  if (!a->q || !a->kv || !a->o) return fail(PA_ERR_NULL, "pa_attn_core: q/kv/o must be non-NULL");
  if (a->G <= 0 || a->H <= 0 || a->n_q <= 0 || a->n_k <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_attn_core: G,H,n_q,n_k must be positive");
  AttnLaunch l = {};
  l.hd = a->head_dim ? a->head_dim : 64;
  l.windowed = false;
  l.G = a->G; l.H = a->H; l.n_q = a->n_q; l.n_k = a->n_k;
  l.q = a->q; l.ldq = a->ldq; l.q_group = a->q_group; l.q_col0 = a->q_col0;
  l.k = a->kv; l.v = a->kv; l.ldk = a->ldkv; l.k_group = a->kv_group; l.k_col0 = a->k_col0; l.v_col0 = a->v_col0;
  l.o = a->o; l.ldo = a->ldo; l.o_group = a->o_group; l.o_col0 = a->o_col0;
  l.scale = a->scale;
  return attn_launch(l, st);
}

// LayerNorm row kernel: the instantiation that holds exactly the row's width in registers (C <= 1024), else the generic kernel
void launch_layernorm(const LnParams& ln, cudaStream_t st) {
  const int blocks = (int)((ln.rows * 32 + 255) / 256);
  if (ln.C % 8 == 0 && ln.C <= 256) layernorm_rows_kernel<1><<<blocks, 256, 0, st>>>(ln);
  else if (ln.C % 8 == 0 && ln.C <= 512) layernorm_rows_kernel<2><<<blocks, 256, 0, st>>>(ln);
  else if (ln.C % 8 == 0 && ln.C <= 768) layernorm_rows_kernel<3><<<blocks, 256, 0, st>>>(ln);
  else if (ln.C % 8 == 0 && ln.C <= 1024) layernorm_rows_kernel<4><<<blocks, 256, 0, st>>>(ln);
  else layernorm_kernel<<<blocks, 256, 0, st>>>(ln);
}

int grid_for(long long work_items, int threads) {
  long long blocks = (work_items + threads - 1) / threads;
  const long long cap = (long long)num_sms() * 16;
  return (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}

}  // namespace

// ------------------------------------------------------------------------------------------------ exports
// tile width of a GEMM phase of the fused kernel: the cost model of pick_block_n restricted to the instantiated widths
static int fused_pick_bn(int M, int N, int K) {
  const int workers = num_sms() / 2, m_tiles = (M + 255) / 256, num_kb = (K + 63) / 64;
  double best = 1e30;
  int best_bn = 256;
  const int cands[2] = {256, 192};
  for (int i = 0; i < 2; ++i) {
    const int bn = cands[i];
    const long long tiles = (long long)m_tiles * ((N + bn - 1) / bn);
    // inside the fused kernel a partial last wave is mostly absorbed by the next phase: charge the exact average plus
    // half a tile for the remainder instead of whole waves
    const double per_tile = 2.0 * num_kb * bn + 700.0;
    const double cost = ((double)tiles / workers + (tiles % workers ? 0.5 : 0.0)) * per_tile;
    if (cost < best * 0.999) { best = cost; best_bn = bn; }
  }
  return best_bn;
}

template <int BN1, int BN2>
static int launch_vit_fused(const GemmPlan& p1, const AttnPlan& pa_, const GemmPlan& p2, const VitFusedParams& fp, int smem, cudaStream_t st) {
  static SmemAttr smem_attr;
  { const int rc = smem_attr.ensure(vit_fused_kernel<BN1, BN2>, smem); if (rc) return rc; }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((num_sms() / 2) * 2);
  cfg.blockDim = dim3(ATTN_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  {
    // the phases spin-wait on each other across SMs: launch only a grid the device can hold at once (one CTA per SM; for
    // this one-CTA-per-SM kernel the occupancy calculator's answer is exact), else let the caller use three launches
    static std::mutex mu;
    static int resident[64];
    static int resident_smem[64];
    int dev = 0;
    cudaGetDevice(&dev);
    dev &= 63;
    std::lock_guard<std::mutex> lk(mu);
    if (resident_smem[dev] != smem) {
      int n = 0;
      PA_CUDA_OK(cudaOccupancyMaxActiveClusters(&n, vit_fused_kernel<BN1, BN2>, &cfg));
      resident[dev] = n; resident_smem[dev] = smem;
    }
    if (resident[dev] < (int)cfg.gridDim.x / 2) return 1;
  }
  PA_CUDA_OK(cudaLaunchKernelEx(&cfg, vit_fused_kernel<BN1, BN2>, p1.tmA, p1.tmB, p1.tmD, pa_.tq, pa_.tk, pa_.tv, pa_.to, p2.tmA, p2.tmB,
                                p2.tmD, fp));
  return PA_OK;
}


// Co-scheduled single launch (pa_cosched.cuh): 2 CTAs per SM in clusters of 2.  Returns 1 when the configuration cannot be
// guaranteed fully co-resident on this device (the caller then uses the sequenced kernel), 0 on success, < 0 on error.
// cudaOccupancyMaxActiveClusters cannot answer the question: for any kernel that executes tcgen05.alloc it reports one CTA per
// SM (measured on B200 / CUDA 12.9: tools/occ_probe.cu), although two CTAs that allocate 256 TMEM columns each are placed
// on every SM.  So residency is established once per device and shared-memory size by the kernel itself in probe mode
// (no work: every CTA allocates its TMEM, announces itself and waits up to ~5 ms to see the whole grid) -- one launch and
// one stream synchronisation at the first qualifying call; never inside a stream capture (that call takes the other path).
static int launch_vit_cosched(const GemmPlan& p1, const CUtensorMap& tmD1, const AttnPlan& pa_, const GemmPlan& p2, const CUtensorMap& tmD2,
                              const CUtensorMap& tmB1q, const CUtensorMap& tmB2q, CsParams cp, int smem, cudaStream_t st) {
  struct DevState { int smem_set = 0; int probed_smem = 0; int resident = 0; };
  static DevState state[64];
  static std::mutex mu;
  int dev = 0;
  cudaGetDevice(&dev);
  dev &= 63;
  const int grid = (num_sms() / 2) * 4;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(CS_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  {
    std::lock_guard<std::mutex> lk(mu);
    DevState& ds = state[dev];
    if (ds.smem_set < smem) {
      PA_CUDA_OK(cudaFuncSetAttribute(vit_cosched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      PA_CUDA_OK(cudaFuncSetAttribute(vit_cosched_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      ds.smem_set = smem;
    }
    if (ds.probed_smem < smem) {
      cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
      PA_CUDA_OK(cudaStreamIsCapturing(st, &cap));
      if (cap != cudaStreamCaptureStatusNone) return 1;           // cannot synchronise here: not established yet
      // the scheduling words were zeroed by the caller's memset on this stream; the probe counters live behind them
      CsParams pp = cp;
      pp.probe = cp.sched + cs_sched_ints(grid);
      PA_CUDA_OK(cudaMemsetAsync(pp.probe, 0, 2 * sizeof(int), st));
      PA_CUDA_OK(cudaLaunchKernelEx(&cfg, vit_cosched_kernel, p1.tmA, p1.tmB, tmD1, pa_.tq, pa_.tk, pa_.tv, pa_.to, p2.tmA, p2.tmB, tmD2, tmB1q, tmB2q, pp));
      int seen[2] = {0, 0};
      PA_CUDA_OK(cudaMemcpyAsync(seen, pp.probe, sizeof(seen), cudaMemcpyDeviceToHost, st));
      PA_CUDA_OK(cudaStreamSynchronize(st));
      ds.probed_smem = smem;
      ds.resident = (seen[1] == grid);
      // the probe launch consumed the role tickets: zero them again for the real launch
      PA_CUDA_OK(cudaMemsetAsync(cp.sched, 0, (size_t)cs_sched_ints(grid) * sizeof(int), st));
    }
    if (!ds.resident) {
      fail(PA_ERR_UNSUPPORTED, "co-scheduled kernel: the residency probe did not see %d CTAs (2 per SM) resident at once (dynamic smem %d B)", grid, smem);
      return 1;
    }
  }
  cp.probe = nullptr;
  PA_CUDA_OK(cudaLaunchKernelEx(&cfg, vit_cosched_kernel, p1.tmA, p1.tmB, tmD1, pa_.tq, pa_.tk, pa_.tv, pa_.to, p2.tmA, p2.tmB, tmD2, tmB1q, tmB2q, cp));
  return PA_OK;
}

// LePEAttention as ONE kernel (pa_attn_win.cuh: window-resident Q/K/V, LePE in the epilogue).  Returns 1 when the window does not
// fit the two-CTAs-per-SM shared-memory plan (the caller then runs the LePE kernel + the windowed two-slot core).
template <int HD>
static int launch_attn_win(const AttnPlan& plan, const pa_cswin_lepe_args* a, cudaStream_t st) {
  AttnWinParams wp = {};
  wp.at = plan.p;
  wp.at.add_into_out = 0;
  wp.lepe_w = a->get_v_weight_t; wp.lepe_b = a->get_v_bias; wp.Cb = a->C;
  wp.q_rows = attn_win_q_rows(plan.p.q_tiles, plan.p.nkb, plan.p.kb_rows);
  wp.kv_rows = attn_win_kv_rows(plan.p.nkb, plan.p.kb_rows, plan.p.kb);
  if (plan.p.nkb > 1 && plan.p.kb > 256 - HD) return 1;
  const int smem = attn_win_data_bytes(HD, wp.q_rows, wp.kv_rows, a->C) + 64 + 1024;
  if (smem > 115712) return 1;
  static SmemAttr smem_attr;
  int rc = smem_attr.ensure(attn_win_kernel<HD>, smem);
  if (rc) return rc;
  {
    static std::mutex mu;
    static bool carve[64];
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(mu);
    if (!carve[dev & 63]) {
      PA_CUDA_OK(cudaFuncSetAttribute(attn_win_kernel<HD>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
      carve[dev & 63] = true;
    }
  }
  const int units = plan.p.G * plan.p.H;
  const int cap = 2 * num_sms();
  attn_win_kernel<HD><<<units < cap ? units : cap, CS_THREADS, smem, st>>>(plan.tq, plan.tk, plan.tv, wp);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return PA_OK;
}


extern "C" {

int pa_version(void) { return PA_VERSION; }
const char* pa_last_error(void) { return err_buf(); }
unsigned long long pa_launch_count(void) { return launch_counter().load(); }

int pa_device_check(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) return fail(PA_ERR_DEVICE, "no CUDA device (this library has no CPU fallback)");
  if (device < 0 || device >= n) return fail(PA_ERR_DEVICE, "device %d out of range (count %d)", device, n);
  int major = 0;
  PA_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) return fail(PA_ERR_DEVICE, "device %d is compute capability %d.x; sm_100 (B200) required", device, major);
  return PA_OK;
}

/* debug: device buffer of >= 64*8 int64 that CTA 0 of every later GEMM launch fills with clock64 stamps (NULL = off) */
void pa_debug_set_gemm_trace(void* device_buffer) { g_gemm_trace = reinterpret_cast<long long*>(device_buffer); }

int pa_gemm_tn(const pa_gemm_args* a, void* stream) { return gemm_impl(a, (cudaStream_t)stream); }

int pa_cast_f32(const float* src, void* dst, long long n, int out_dtype, void* stream) {
  if (!src || !dst) return fail(PA_ERR_NULL, "pa_cast_f32: src/dst must be non-NULL");
  if (n < 0) return fail(PA_ERR_BAD_SHAPE, "pa_cast_f32: n must be >= 0");
  if (out_dtype != PA_DTYPE_F16 && out_dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "pa_cast_f32: out_dtype must be fp16/bf16");
  if ((reinterpret_cast<uintptr_t>(src) & 15) || (reinterpret_cast<uintptr_t>(dst) & 15)) return fail(PA_ERR_MISALIGNED, "pa_cast_f32: buffers must be 16-byte aligned");
  int rc = current_device_check();
  if (rc) return rc;
  if (n == 0) return PA_OK;
  const long long n8 = n / 8;
  const int tail = (int)(n - n8 * 8);
  cast_f32_to_16_kernel<<<grid_for(n8 > 0 ? n8 : 1, 256), 256, 0, (cudaStream_t)stream>>>(
      reinterpret_cast<const float4*>(src), reinterpret_cast<uint4*>(dst), n8, out_dtype == PA_DTYPE_BF16, src + n8 * 8,
      reinterpret_cast<uint16_t*>(dst) + n8 * 8, tail);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return PA_OK;
}
int pa_attn_core(const pa_attn_args* a, void* stream) { return attn_impl(a, (cudaStream_t)stream); }

// ================================================================ ViT  (ViT.py:67-89)
static int vit_check(const pa_vit_args* a) {
  if (!a) return fail(PA_ERR_NULL, "pa_vit: args is NULL");
  if (a->B <= 0 || a->N <= 0 || a->C <= 0 || a->H <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_vit: B,N,C,H must be positive");
  if (a->C % a->H != 0) return fail(PA_ERR_BAD_SHAPE, "pa_vit: dim %d not divisible by num_heads %d (ViT.py:70)", a->C, a->H);
  if (!attn_hd_ok(a->C / a->H)) return fail(PA_ERR_UNSUPPORTED, "pa_vit: head_dim %d unsupported (multiples of 16 from 32 to 192)", a->C / a->H);
  if (a->dtype != PA_DTYPE_F16 && a->dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "pa_vit: dtype must be fp16/bf16");
  return PA_OK;
}

static int vit_three_launches(const pa_vit_args* a, const void* x_in, int x_dtype, const void* residual, void* qkv, void* obuf, cudaStream_t st,
                              float* knn_thresh = nullptr);

// dependency counters (per 128-row tile of qkv + per image) followed by the co-scheduled kernel's scheduling words
static size_t vit_counter_ints(const pa_vit_args* a) {
  const size_t rows = (size_t)a->B * a->N;
  return (rows + 127) / 128 + a->B + cs_sched_ints(4 * 1024) + 2;
}

size_t pa_vit_workspace_bytes(const pa_vit_args* a) {
  if (vit_check(a)) return 0;
  const size_t rows = (size_t)a->B * a->N;
  return align_up(rows * 3 * a->C * 2, 1024) + align_up(rows * a->C * 2, 1024) + align_up(vit_counter_ints(a) * 4, 1024) +
         (a->topk > 0 ? align_up(rows * a->H * 4, 1024) : 0) + 1024;
}

int pa_vit_fwd(const pa_vit_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = vit_check(a);
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->proj_weight || !a->y) return fail(PA_ERR_NULL, "pa_vit_fwd: x/qkv_weight/proj_weight/y must be non-NULL");
  const size_t need = pa_vit_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_vit_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)a->B * a->N;
  const int C = a->C;
  Arena ws(workspace);
  void* qkv = ws.take((size_t)rows * 3 * C * 2);
  void* obuf = ws.take((size_t)rows * C * 2);
  int* counters = reinterpret_cast<int*>(ws.take(vit_counter_ints(a) * sizeof(int)));
  const int n_mt = (int)((rows + 127) / 128);
  const EnvCfg& ev = env();
  // ---- single-launch paths.  Default whenever the shape qualifies: the co-scheduled kernel (pa_cosched.cuh: projection
  //      GEMMs under the softmax chain, two role-specialised CTAs per SM), else the sequenced kernel (pa_fused.cuh: the three
  //      phases back to back per SM).  PA_VIT_FUSED=0 selects three launches, =1 makes a shape no single-launch kernel
  //      takes an error instead of a silent switch; PA_VIT_COSCHED=0 / 1 never / always takes the co-scheduled kernel.
  const int hd = C / a->H;
  if (a->topk != 0) {
    // kvt.KNNAttention (kvt.py:67-94): qkv GEMM -> per-row k-th largest score -> attention core with the row threshold -> proj GEMM
    if (a->topk < 0 || a->topk > a->N) return fail(PA_ERR_BAD_SHAPE, "pa_vit_fwd: topk=%d must lie in [1, N=%d] (torch.topk, kvt.py:85)", a->topk, a->N);
    if (hd != 64 || a->N > 240) return fail(PA_ERR_UNSUPPORTED, "pa_vit_fwd(topk): needs 64-wide heads and N <= 240 (got head_dim %d, N=%d)", hd, a->N);
    if ((rc = current_device_check())) return rc;
    float* thr = reinterpret_cast<float*>(ws.take((size_t)rows * a->H * 4));
    return vit_three_launches(a, a->x, a->dtype, nullptr, qkv, obuf, st, thr);
  }
  const bool fused_forced = ev.vit_fused > 0 || ev.vit_cosched > 0;
  const bool fused_wanted = ev.vit_fused != 0;
  bool fused_ok = fused_wanted && a->N <= 256 && hd == 64;
  if (fused_forced && !fused_ok)
    return fail(PA_ERR_UNSUPPORTED, "pa_vit_fwd(single launch): needs N <= 256 (one key block) and 64-wide heads; got N=%d, head_dim=%d", a->N, hd);
  if (fused_ok) {
    if ((rc = current_device_check())) return rc;
    pa_gemm_args g1 = {};
    g1.a_dtype = a->dtype; g1.b_dtype = a->dtype; g1.out_dtype = PA_DTYPE_F16;
    g1.M = (int)rows; g1.N = 3 * C; g1.K = C; g1.Z = 1;
    g1.A = a->x; g1.lda = C; g1.B = a->qkv_weight; g1.ldb = C; g1.D = qkv; g1.ldd = 3 * C;
    g1.bias = a->qkv_bias; g1.bias_mode = a->qkv_bias ? 1 : 0;
    pa_gemm_args g2 = {};
    g2.a_dtype = PA_DTYPE_F16; g2.b_dtype = PA_DTYPE_F16; g2.out_dtype = a->out_dtype;
    g2.M = (int)rows; g2.N = C; g2.K = C; g2.Z = 1;
    g2.A = obuf; g2.lda = C; g2.B = a->proj_weight; g2.ldb = C; g2.D = a->y; g2.ldd = C;
    g2.bias = a->proj_bias; g2.bias_mode = a->proj_bias ? 1 : 0;
    AttnLaunch al = {};
    al.hd = 64; al.G = a->B; al.H = a->H; al.n_q = a->N; al.n_k = a->N;
    al.q = qkv; al.ldq = 3 * C; al.q_group = (long long)a->N * 3 * C; al.q_col0 = 0;
    al.k = qkv; al.v = qkv; al.ldk = 3 * C; al.k_group = (long long)a->N * 3 * C; al.k_col0 = C; al.v_col0 = 2 * C;
    al.o = obuf; al.ldo = C; al.o_group = (long long)a->N * C; al.o_col0 = 0;
    al.scale = a->scale;
    AttnPlan pa_;
    if ((rc = attn_prepare(al, &pa_))) return rc;
    const int grid_cs = (num_sms() / 2) * 4;
    // ---------------- co-scheduled kernel
    bool cs_ok = ev.vit_cosched != 0 && pa_.p.tma_store && pa_.p.kb <= 240 && C % 64 == 0 && a->out_dtype != PA_DTYPE_F32 &&
                 cs_smem_bytes(pa_.p.kb) <= 112 * 1024 && grid_cs <= 4 * 1024;
    if (ev.vit_cosched > 0 && !cs_ok)
      return fail(PA_ERR_UNSUPPORTED, "pa_vit_fwd(co-scheduled): needs N <= 240, dim %% 64 == 0, a 16-bit y and 16-byte aligned buffers");
    if (cs_ok) {
      GemmPlan p1, p2;
      if ((rc = gemm_prepare(&g1, &p1, 256, -2))) return rc;
      if ((rc = gemm_prepare(&g2, &p2, 256, -2))) return rc;
      CUtensorMap tmD1, tmD2;                 // per-warp output boxes: 32 columns x 32 rows, 64-byte swizzle
      {
        uint64_t dims[3] = {(uint64_t)(3 * C), (uint64_t)rows, 1};
        uint64_t str[2] = {(uint64_t)(3 * C) * 2, (uint64_t)(3 * C) * 2 * (uint64_t)rows};
        uint32_t box[3] = {32, 32, 1};
        if ((rc = make_tmap_16b(&tmD1, PA_DTYPE_F16, qkv, 3, dims, str, box, TM_SWZ_64))) return rc;
      }
      if (p2.p.tma_store) {
        uint64_t dims[3] = {(uint64_t)C, (uint64_t)rows, 1};
        uint64_t str[2] = {(uint64_t)C * 2, (uint64_t)C * 2 * (uint64_t)rows};
        uint32_t box[3] = {32, 32, 1};
        if ((rc = make_tmap_16b(&tmD2, a->out_dtype, a->y, 3, dims, str, box, TM_SWZ_64))) return rc;
      } else {
        cs_ok = false;
      }
      if (cs_ok) {
        CsParams cp = {};
        const GemmPlan* gp[2] = {&p1, &p2};
        for (int i = 0; i < 2; ++i) {
          CsGemmPhase& g = cp.g[i];
          g.M = gp[i]->p.M; g.N = gp[i]->p.N;
          g.m_tiles = gp[i]->p.m_tiles; g.m_groups = (g.m_tiles + 1) / 2; g.n_tiles = (g.N + CS_BN - 1) / CS_BN;
          g.tiles = g.m_groups * g.n_tiles;
          g.bias = gp[i]->p.bias; g.out_dtype = gp[i]->p.out_dtype; g.idesc = gp[i]->p.idesc;
        }
        cp.K = C;
        {
          // tile order of the GEMM stream: all qkv tiles first, then the proj tiles (lag = m_groups).  Interleaving the proj
          // tiles of early images (PA_CS_LAG = how many m-groups they trail their rows' qkv tiles) was measured and is WORSE:
          // ViT-B 86 us at lag 50 (= all first), 95 at 18, 123 at 9, 199 at 1 -- the attention stream runs behind the qkv
          // production, a proj tile that waits for it stalls its worker's later qkv tiles, and that starves the attention further
          const int MG = cp.g[0].m_groups;
          int lag = ev.cs_lag > 0 ? ev.cs_lag : MG;
          cp.lag = lag < 1 ? 1 : lag > MG ? MG : lag;
        }
        // tail split (cs_tile): the proj tiles of the last m-groups as 256 x 64 quarters; their B boxes hold 32 rows per CTA
        CUtensorMap tmB1q, tmB2q;
        {
          uint64_t dims[3] = {(uint64_t)C, (uint64_t)C, 1};
          uint64_t str[2] = {(uint64_t)C * 2, (uint64_t)C * C * 2};
          uint32_t box[3] = {64, 32, 1};
          if ((rc = make_tmap_16b(&tmB2q, PA_DTYPE_F16, a->proj_weight, 3, dims, str, box))) return rc;
          uint64_t dims1[3] = {(uint64_t)C, (uint64_t)(3 * C), 1};
          uint64_t str1[2] = {(uint64_t)C * 2, (uint64_t)C * 3 * C * 2};
          if ((rc = make_tmap_16b(&tmB1q, a->dtype, a->qkv_weight, 3, dims1, str1, box))) return rc;
        }
        {
          const int MG = cp.g[0].m_groups;
          // measured (tools/cosched_tail_sweep.py, profiles/cosched_tail_sweep_r02.txt): ViT-B (K = 768) 85.9 us at tail 0, 84.0-84.5 at
          // 3-4, no gain beyond; ViT-L (K = 1024) 119 us at 0, 121-134 with any tail (the quarter tiles' port-bound mainloop is
          // twice as long there) -> four m-groups for K <= 768, none above
          int tail = ev.cs_tail >= 0 ? ev.cs_tail : (C <= 768 ? 4 : 0);
          if (cp.lag != MG) tail = 0;
          if (tail > MG) tail = MG;
          cp.tail = tail;
          cp.g[1].tiles = (MG - tail) * cp.g[1].n_tiles + tail * cp.g[1].n_tiles * (CS_BN / 64);
          int qtail = ev.cs_qtail >= 0 ? ev.cs_qtail : 0;
          if (cp.lag != MG) qtail = 0;
          if (qtail > MG) qtail = MG;
          cp.qtail = qtail;
          cp.g[0].tiles = (MG - qtail) * cp.g[0].n_tiles + qtail * cp.g[0].n_tiles * (CS_BN / 64);
        }
        cp.d[0] = qkv; cp.d[1] = a->y;
        cp.at = pa_.p;
        cp.g[0].signal_ctr = counters;                       // per 128-row tile of qkv: every epilogue warp of every column tile
        cp.at.wait_ctr = counters; cp.at.wait_target = cp.g[0].n_tiles * CS_EPI_WARPS * (CS_BN / 64);   // a full tile's warp publishes 4, a quarter's 1
        cp.at.wait_rows_per_group = a->N;
        cp.at.signal_ctr = counters + n_mt;                  // per image: one count per (head, query tile)
        cp.g[1].wait_ctr = counters + n_mt; cp.g[1].wait_rows = a->N; cp.g[1].wait_target = a->H * cp.at.q_tiles;
        cp.sched = counters + n_mt + a->B;
        cp.trace = g_gemm_trace;
        cp.debug = ev.cs_debug;
        if (cp.debug & 1) cp.g[1].wait_ctr = nullptr;       // experiments: the idle role's dependants must not wait for it
        if (cp.debug & 2) cp.at.wait_ctr = nullptr;
        PA_CUDA_OK(cudaMemsetAsync(counters, 0, (size_t)(n_mt + a->B + cs_sched_ints(grid_cs)) * sizeof(int), st));
        rc = launch_vit_cosched(p1, tmD1, pa_, p2, tmD2, tmB1q, tmB2q, cp, cs_smem_bytes(pa_.p.kb) + 1024, st);
        if (rc < 0) return rc;
        if (rc == 0) { launch_counter()++; t_last_vit_path = 3; return PA_OK; }
        if (ev.vit_cosched > 0) return PA_ERR_UNSUPPORTED;    // message set by launch_vit_cosched
      }
    }
    // ---------------- sequenced kernel
    if (!pa_.p.tma_store) {
      if (fused_forced) return fail(PA_ERR_UNSUPPORTED, "pa_vit_fwd(fused): staged attention epilogue does not fit");
      fused_ok = false;
    }
    GemmPlan p1, p2;
    int bn1 = fused_pick_bn((int)rows, 3 * C, C), bn2 = fused_pick_bn((int)rows, C, C);
    if (ev.fused_bn1 == 192 || ev.fused_bn1 == 256) bn1 = ev.fused_bn1;     // experiments
    if (ev.fused_bn2 == 192 || ev.fused_bn2 == 256) bn2 = ev.fused_bn2;
    if ((rc = gemm_prepare(&g1, &p1, bn1, -2))) return rc;
    if ((rc = gemm_prepare(&g2, &p2, bn2, -2))) return rc;
    const int smem = bn1 == 256 ? (bn2 == 256 ? vit_fused_smem_bytes<256, 256>(pa_.p.kb) : vit_fused_smem_bytes<256, 192>(pa_.p.kb))
                                : (bn2 == 256 ? vit_fused_smem_bytes<192, 256>(pa_.p.kb) : vit_fused_smem_bytes<192, 192>(pa_.p.kb));
    if (!p1.p.tma_store || !p2.p.tma_store || smem > 227 * 1024) {
      if (fused_forced) return fail(PA_ERR_UNSUPPORTED, "pa_vit_fwd(fused): outputs must be TMA-storable and the plan (%d B) must fit", smem);
      fused_ok = false;
    }
    if (fused_ok) {
      PA_CUDA_OK(cudaMemsetAsync(counters, 0, (size_t)(n_mt + a->B) * sizeof(int), st));
      VitFusedParams fp;
      fp.g1 = p1.p; fp.at = pa_.p; fp.g2 = p2.p;
      fp.g1.m_groups = (fp.g1.m_tiles + 1) / 2; fp.g1.balanced = 0;
      fp.g2.m_groups = (fp.g2.m_tiles + 1) / 2; fp.g2.balanced = 0;
      if (g_gemm_trace) { fp.g1.trace = g_gemm_trace; fp.at.trace = g_gemm_trace + 512; fp.g2.trace = g_gemm_trace + 1024; }
      {
        // static balance: each phase's remainder units (the CTAs that get one unit more than the others) are placed on
        // different CTAs -- qkv extras on pairs [0, r1), attention extras on the CTAs after them, and the proj phase
        // rotated so that its light pairs are the ones that were heavy before
        const int grid = (num_sms() / 2) * 2, ncl = grid / 2;
        const int r1 = (fp.g1.m_groups * fp.g1.n_tiles) % ncl;
        const int r3 = (fp.g2.m_groups * fp.g2.n_tiles) % ncl;
        fp.at.cta_shift = (2 * r1) % grid;
        fp.g2.worker_shift = r3;
      }
      fp.g1.signal_ctr = counters;                                   // per 128-row tile of qkv
      fp.at.wait_ctr = counters; fp.at.wait_target = fp.g1.n_tiles * FUSED_ESETS;   // every epilogue set of every column tile publishes
      fp.at.wait_rows_per_group = a->N;
      fp.at.signal_ctr = counters + n_mt;                            // per image
      fp.g2.wait_ctr = counters + n_mt; fp.g2.wait_rows = a->N; fp.g2.wait_target = a->H * fp.at.q_tiles;
      if (bn1 == 256 && bn2 == 192) rc = launch_vit_fused<256, 192>(p1, pa_, p2, fp, smem, st);
      else if (bn1 == 256) rc = launch_vit_fused<256, 256>(p1, pa_, p2, fp, smem, st);
      else if (bn2 == 256) rc = launch_vit_fused<192, 256>(p1, pa_, p2, fp, smem, st);
      else rc = launch_vit_fused<192, 192>(p1, pa_, p2, fp, smem, st);
      if (rc < 0) return rc;
      if (rc == 0) {
        launch_counter()++;
        t_last_vit_path = 2;
        return PA_OK;
      }
      if (fused_forced) return fail(PA_ERR_UNSUPPORTED, "pa_vit_fwd(fused): the device cannot hold one CTA of the kernel on every SM at once");
    }
  }
  t_last_vit_path = 1;
  // ---- three launches (any N, any supported head dim; also the reference point the single-launch kernels are tested against)
  return vit_three_launches(a, a->x, a->dtype, nullptr, qkv, obuf, st);
}

// qkv GEMM -> attention core -> proj GEMM (+ residual in its epilogue).  x_in: the qkv GEMM's A operand (a->x, or the LayerNorm
// output of the block entry point); residual: nullptr or the tensor added to proj's result (dtype a->dtype, pitch C).
static int vit_three_launches(const pa_vit_args* a, const void* x_in, int x_dtype, const void* residual, void* qkv, void* obuf, cudaStream_t st,
                              float* knn_thresh) {
  int rc;
  const long long rows = (long long)a->B * a->N;
  const int C = a->C, hd = C / a->H;
  // 1. qkv[B*N, 3C] = x Wqkv^T (+b)          (ViT.py:81)
  if ((rc = linear(x_in, x_dtype, C, a->qkv_weight, x_dtype, a->qkv_bias, qkv, PA_DTYPE_F16, 3 * C, rows, 3 * C, C, st))) return rc;
  // 2. per (b,h): softmax(q k^T scale) v       (ViT.py:83-86), O as [B*N, C] with column h*hd+d
  AttnLaunch at = {};
  at.hd = hd; at.G = a->B; at.H = a->H; at.n_q = a->N; at.n_k = a->N;
  at.q = qkv; at.ldq = 3 * C; at.q_group = (long long)a->N * 3 * C; at.q_col0 = 0;
  at.k = qkv; at.v = qkv; at.ldk = 3 * C; at.k_group = (long long)a->N * 3 * C; at.k_col0 = C; at.v_col0 = 2 * C;
  at.o = obuf; at.ldo = C; at.o_group = (long long)a->N * C; at.o_col0 = 0;
  at.scale = a->scale;
  if (knn_thresh != nullptr) {
    // kvt.py:84-87: the k-th largest raw score of every row (scale > 0 keeps the order)
    KnnParams kp;
    kp.qkv = qkv; kp.thresh = knn_thresh; kp.G = a->B; kp.H = a->H; kp.N = a->N; kp.hd = hd; kp.topk = a->topk;
    kp.ld = 3 * C; kp.group = (long long)a->N * 3 * C; kp.q_col0 = 0; kp.k_col0 = C;
    const long long warps = rows * a->H;
    knn_threshold_kernel<8><<<(int)((warps * 32 + 255) / 256), 256, 0, st>>>(kp);      // N <= 240 < 256 keys
    PA_CUDA_OK(cudaGetLastError());
    launch_counter()++;
    at.row_thresh = knn_thresh;
  }
  if ((rc = attn_launch(at, st))) return rc;
  // 3. y = O Wproj^T + b (+ residual)          (ViT.py:87, :116)
  return linear(obuf, PA_DTYPE_F16, C, a->proj_weight, PA_DTYPE_F16, a->proj_bias, a->y, a->out_dtype, C, rows, C, C, st,
                residual, C, a->dtype);
}

// ================================================================ ViT block, attention half  (ViT.py:116)
size_t pa_vit_block_attn_workspace_bytes(const pa_vit_block_args* a) {
  if (!a || vit_check(&a->attn)) return 0;
  const size_t rows = (size_t)a->attn.B * a->attn.N;
  return align_up(rows * a->attn.C * 2, 1024) + pa_vit_workspace_bytes(&a->attn);
}

int pa_vit_block_attn_fwd(const pa_vit_block_args* b, void* workspace, size_t workspace_bytes, void* stream) {
  if (!b) return fail(PA_ERR_NULL, "pa_vit_block_attn_fwd: args is NULL");
  const pa_vit_args* a = &b->attn;
  int rc = vit_check(a);
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->proj_weight || !a->y || !b->ln_weight || !b->ln_bias)
    return fail(PA_ERR_NULL, "pa_vit_block_attn_fwd: x/qkv_weight/proj_weight/y/ln_weight/ln_bias must be non-NULL");
  if (a->C % 8) return fail(PA_ERR_BAD_SHAPE, "pa_vit_block_attn_fwd: dim must be a multiple of 8");
  const size_t need = pa_vit_block_attn_workspace_bytes(b);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_vit_block_attn_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)a->B * a->N;
  const int C = a->C;
  Arena ws(workspace);
  void* img = ws.take((size_t)rows * C * 2);
  void* qkv = ws.take((size_t)rows * 3 * C * 2);
  void* obuf = ws.take((size_t)rows * C * 2);
  // img = layernorm1(x)   (ViT.py:116), fp16
  LnParams ln;
  ln.x = a->x; ln.out = img; ln.gamma = b->ln_weight; ln.beta = b->ln_bias; ln.rows = rows; ln.C = C; ln.dtype = a->dtype; ln.eps = b->ln_eps;
  launch_layernorm(ln, st);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  // x + proj(attention(img)): the residual rides in the proj GEMM's epilogue
  return vit_three_launches(a, img, PA_DTYPE_F16, a->x, qkv, obuf, st);
}

/* debug: occupancy facts of the co-scheduled kernel for `smem` bytes of dynamic shared memory; out[0..5] = registers per thread,
 * static shared bytes, resident blocks per SM (plain launch), resident clusters of 2 (device-wide), max threads per block,
 * binary version */
int pa_debug_cosched_occupancy(int smem, int* out) {
  cudaFuncAttributes fa;
  PA_CUDA_OK(cudaFuncGetAttributes(&fa, vit_cosched_kernel));
  PA_CUDA_OK(cudaFuncSetAttribute(vit_cosched_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  PA_CUDA_OK(cudaFuncSetAttribute(vit_cosched_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
  int nb = -1, nc = -1;
  PA_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, vit_cosched_kernel, CS_THREADS, smem));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((num_sms() / 2) * 4); cfg.blockDim = dim3(CS_THREADS); cfg.dynamicSmemBytes = smem;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  PA_CUDA_OK(cudaOccupancyMaxActiveClusters(&nc, vit_cosched_kernel, &cfg));
  out[0] = fa.numRegs; out[1] = (int)fa.sharedSizeBytes; out[2] = nb; out[3] = nc; out[4] = fa.maxThreadsPerBlock; out[5] = fa.binaryVersion;
  return PA_OK;
}

/* which path the calling thread's last successful pa_vit_fwd took: 1 three launches, 2 sequenced single launch, 3 co-scheduled
 * single launch (0: none yet) */
int pa_last_vit_path(void) { return t_last_vit_path; }

/* re-read the PA_* environment switches (they are cached at the first call) */
void pa_reload_env(void) {
  std::lock_guard<std::mutex> lk(g_env_mu);
  g_env.store(env_load(), std::memory_order_release);
}

// ================================================================ BViT  (bvit.py:49-76)
static int bvit_check(const pa_bvit_args* a) {
  if (!a) return fail(PA_ERR_NULL, "pa_bvit: args is NULL");
  if (a->B <= 0 || a->N <= 0 || a->C <= 0 || a->H <= 0 || a->dim_head <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_bvit: B,N,C,H,dim_head must be positive");
  if (!attn_hd_ok(a->dim_head)) return fail(PA_ERR_UNSUPPORTED, "pa_bvit: dim_head %d unsupported (multiples of 16 from 32 to 192)", a->dim_head);
  if (a->C % 8) return fail(PA_ERR_BAD_SHAPE, "pa_bvit: dim must be a multiple of 8");
  if (a->dtype != PA_DTYPE_F16 && a->dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "pa_bvit: dtype must be fp16/bf16");
  if (!a->out_weight && (a->H * a->dim_head != a->C || a->out_dtype != PA_DTYPE_F16))
    return fail(PA_ERR_UNSUPPORTED, "pa_bvit: without an output projection the inner width must equal dim and y must be fp16");
  return PA_OK;
}

size_t pa_bvit_workspace_bytes(const pa_bvit_args* a) {
  if (bvit_check(a)) return 0;
  return align_up((size_t)a->B * a->N * a->H * a->dim_head * 2, 1024) + 1024;
}

int pa_bvit_fwd(const pa_bvit_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = bvit_check(a);
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->qkv || !a->y) return fail(PA_ERR_NULL, "pa_bvit_fwd: x/qkv_weight/qkv/y must be non-NULL");
  const size_t need = pa_bvit_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_bvit_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int C = a->C, inner = a->H * a->dim_head;
  const long long rows = (long long)a->B * a->N;
  Arena ws(workspace);
  void* obuf = a->out_weight ? ws.take((size_t)rows * inner * 2) : a->y;
  // qkv = x Wqkv^T, columns (q|k|v, head, d)          (bvit.py:67-68)
  if ((rc = linear(a->x, a->dtype, C, a->qkv_weight, a->dtype, nullptr, a->qkv, PA_DTYPE_F16, 3 * inner, rows, 3 * inner, C, st))) return rc;
  AttnLaunch at = {};
  at.hd = a->dim_head; at.G = a->B; at.H = a->H; at.n_q = a->N; at.n_k = a->N;
  at.q = a->qkv; at.ldq = 3 * inner; at.q_group = (long long)a->N * 3 * inner; at.q_col0 = 0;
  at.k = a->qkv; at.v = a->qkv; at.ldk = 3 * inner; at.k_group = (long long)a->N * 3 * inner; at.k_col0 = inner; at.v_col0 = 2 * inner;
  at.o = obuf; at.ldo = inner; at.o_group = (long long)a->N * inner; at.o_col0 = 0;
  at.scale = a->scale;
  if ((rc = attn_launch(at, st))) return rc;           // bvit.py:70-75
  if (!a->out_weight) return PA_OK;
  return linear(obuf, PA_DTYPE_F16, inner, a->out_weight, PA_DTYPE_F16, a->out_bias, a->y, a->out_dtype, C, rows, C, inner, st);
}

// ================================================================ PVT  (pvt.py:52-91)
static int pvt_check(const pa_pvt_args* a) {
  if (!a) return fail(PA_ERR_NULL, "pa_pvt: args is NULL");
  if (a->B <= 0 || a->C <= 0 || a->H <= 0 || a->Himg <= 0 || a->Wimg <= 0 || a->sr <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_pvt: sizes must be positive");
  if (a->C % a->H != 0) return fail(PA_ERR_BAD_SHAPE, "pa_pvt: dim %d not divisible by num_heads %d (pvt.py:56)", a->C, a->H);
  if (!attn_hd_ok(a->C / a->H)) return fail(PA_ERR_UNSUPPORTED, "pa_pvt: head_dim %d unsupported (multiples of 16 from 32 to 192)", a->C / a->H);
  if (a->N != a->Himg * a->Wimg) return fail(PA_ERR_BAD_SHAPE, "pa_pvt: N=%d != H*W=%d*%d", a->N, a->Himg, a->Wimg);
  if (a->C % 8) return fail(PA_ERR_BAD_SHAPE, "pa_pvt: dim must be a multiple of 8");
  if (a->dtype != PA_DTYPE_F16 && a->dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "pa_pvt: dtype must be fp16/bf16");
  return PA_OK;
}
static inline int pvt_m(const pa_pvt_args* a) {
  if (a->kv_tokens) return a->kv_count;
  return a->sr > 1 ? (a->Himg / a->sr) * (a->Wimg / a->sr) : a->N;
}

static int pvt_check_full(const pa_pvt_args* a) {
  int rc = pvt_check(a);
  if (rc) return rc;
  if (a->sr_mode != 0 && a->sr_mode != 1) return fail(PA_ERR_BAD_SHAPE, "pa_pvt: sr_mode must be 0 (depthwise + BatchNorm) or 1 (dense conv)");
  if (a->sr > 1 && (a->Himg % a->sr || a->Wimg % a->sr))
    return fail(PA_ERR_BAD_SHAPE, "pa_pvt: H=%d, W=%d not divisible by sr_ratio %d", a->Himg, a->Wimg, a->sr);
  if (a->kv_tokens && (a->sr != 1 || a->kv_count <= 0)) return fail(PA_ERR_BAD_SHAPE, "pa_pvt: kv_tokens needs sr == 1 and kv_count > 0");
  return PA_OK;
}

size_t pa_pvt_workspace_bytes(const pa_pvt_args* a) {
  if (pvt_check_full(a)) return 0;
  const size_t rows = (size_t)a->B * a->N, mrows = (size_t)a->B * pvt_m(a);
  // reduced map, q, attention output, [k|v], and (dense reduction) the patch matrix = a re-partition of x
  return align_up(mrows * a->C * 2, 1024) + align_up(rows * a->C * 2, 1024) * 2 + align_up(mrows * 2 * a->C * 2, 1024) +
         ((a->sr > 1 && a->sr_mode == 1) ? align_up(rows * a->C * 2, 1024) : 0) + 1024;
}

// [sr] -> q GEMM -> [k|v] GEMM -> attention core -> proj GEMM (+ residual in its epilogue).  x_in / x_dtype: the operand of the
// q projection and of the reduction (a->x, or the LayerNorm output of the block entry point); residual: nullptr or the tensor
// added to proj's result (dtype a->dtype, pitch C).  ws: pa_pvt_workspace_bytes(a) bytes.
static int pvt_run(const pa_pvt_args* a, const void* x_in, int x_dtype, const void* residual, void* workspace, cudaStream_t st) {
  int rc;
  const int C = a->C, M = pvt_m(a);
  const long long rows = (long long)a->B * a->N, mrows = (long long)a->B * M;
  Arena ws(workspace);
  void* xr = ws.take((size_t)mrows * C * 2);
  void* qb = ws.take((size_t)rows * C * 2);
  void* ob = ws.take((size_t)rows * C * 2);
  void* kv = ws.take((size_t)mrows * 2 * C * 2);
  const void* kv_in = x_in;
  int kv_dtype = x_dtype;
  if (a->kv_tokens) { kv_in = a->kv_tokens; kv_dtype = PA_DTYPE_F16; }     // p2t: keys / values from the pooled pyramid
  if (a->sr > 1 && a->sr_mode == 0) {
    // spatial reduction: depthwise conv (k = stride = sr) + eval BatchNorm folded into scale/shift   (pvt.py:77-78, cmt.py:97-98)
    SrParams sp;
    sp.x = x_in; sp.out = xr; sp.w = a->sr_weight_t; sp.scale = a->sr_scale; sp.shift = a->sr_shift;
    sp.B = a->B; sp.H = a->Himg; sp.W = a->Wimg; sp.C = C; sp.sr = a->sr; sp.Hs = a->Himg / a->sr; sp.Ws = a->Wimg / a->sr;
    sp.dtype = x_dtype;
    sr_conv_bn_kernel<<<grid_for(mrows * (C / 8), 256), 256, 0, st>>>(sp);
    PA_CUDA_OK(cudaGetLastError());
    launch_counter()++;
    kv_in = xr;
    kv_dtype = PA_DTYPE_F16;
  } else if (a->sr > 1) {
    // spatial reduction: dense conv k = stride = sr (segformer.py:38-39) = GEMM over the sr x sr patches, K = sr*sr*C
    void* patches = ws.take((size_t)rows * C * 2);
    PatchParams pp;
    pp.x = x_in; pp.out = patches; pp.B = a->B; pp.H = a->Himg; pp.W = a->Wimg; pp.C = C; pp.sr = a->sr;
    pp.Hs = a->Himg / a->sr; pp.Ws = a->Wimg / a->sr;
    sr_patchify_kernel<<<grid_for(rows * (C / 8), 256), 256, 0, st>>>(pp);
    PA_CUDA_OK(cudaGetLastError());
    launch_counter()++;
    const int Kd = a->sr * a->sr * C;
    if ((rc = linear(patches, x_dtype, Kd, a->sr_dense_weight, x_dtype, a->sr_dense_bias, xr, PA_DTYPE_F16, C, mrows, C, Kd, st))) return rc;
    kv_in = xr;
    kv_dtype = PA_DTYPE_F16;
  }
  // q = x Wq^T (+b)  (pvt.py:75);  [k|v] = x_ [Wk;Wv]^T (+b)  (pvt.py:79-80 / 82-83, segformer.py:40 / 43)
  if ((rc = linear(x_in, x_dtype, C, a->q_weight, x_dtype, a->q_bias, qb, PA_DTYPE_F16, C, rows, C, C, st))) return rc;
  if ((rc = linear(kv_in, kv_dtype, C, a->kv_weight, kv_dtype, a->kv_bias, kv, PA_DTYPE_F16, 2 * C, mrows, 2 * C, C, st))) return rc;
  AttnLaunch at = {};
  at.hd = C / a->H; at.G = a->B; at.H = a->H; at.n_q = a->N; at.n_k = M;
  at.q = qb; at.ldq = C; at.q_group = (long long)a->N * C; at.q_col0 = 0;
  at.k = kv; at.v = kv; at.ldk = 2 * C; at.k_group = (long long)M * 2 * C; at.k_col0 = 0; at.v_col0 = C;
  at.o = ob; at.ldo = C; at.o_group = (long long)a->N * C; at.o_col0 = 0;
  at.scale = a->scale;
  at.rel_pos = a->rel_pos;                  // cmt.py:100
  // opt-in (PA_PVT_FUSED=1; correct, but measured slower than the two launches: pa_attn_proj.cuh): attention core and
  // projection in ONE kernel for the few-key stages of PVT / SegFormer -- O stays in TMEM
  if (env().pvt_fused && residual == nullptr && attn_proj_ok(at, C, a->out_dtype)) {
    if ((reinterpret_cast<uintptr_t>(a->y) & 15) == 0) return launch_attn_proj(at, a->proj_weight, a->proj_bias, a->y, a->out_dtype, st);
  }
  if ((rc = attn_launch(at, st))) return rc;
  return linear(ob, PA_DTYPE_F16, C, a->proj_weight, PA_DTYPE_F16, a->proj_bias, a->y, a->out_dtype, C, rows, C, C, st,
                residual, C, a->dtype);
}

static int pvt_ptr_check(const pa_pvt_args* a, const char* who) {
  if (!a->x || !a->q_weight || !a->kv_weight || !a->proj_weight || !a->y) return fail(PA_ERR_NULL, "%s: x/weights/y must be non-NULL", who);
  if (a->sr > 1 && a->sr_mode == 0 && (!a->sr_weight_t || !a->sr_scale || !a->sr_shift))
    return fail(PA_ERR_NULL, "%s: sr_ratio>1 needs sr_weight_t/sr_scale/sr_shift", who);
  if (a->sr > 1 && a->sr_mode == 1 && !a->sr_dense_weight) return fail(PA_ERR_NULL, "%s: sr_mode 1 needs sr_dense_weight", who);
  return PA_OK;
}

int pa_pvt_fwd(const pa_pvt_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = pvt_check_full(a);
  if (rc) return rc;
  if ((rc = pvt_ptr_check(a, "pa_pvt_fwd"))) return rc;
  const size_t need = pa_pvt_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_pvt_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  return pvt_run(a, a->x, a->dtype, nullptr, workspace, (cudaStream_t)stream);
}

// ================================================================ P2T  (p2t.py:46-94)
static int p2t_check(const pa_p2t_args* a, int* M_out) {
  if (!a) return fail(PA_ERR_NULL, "pa_p2t: args is NULL");
  int rc = pvt_check(&a->attn);
  if (rc) return rc;
  if (a->attn.sr != 1 || a->attn.sr_mode != 0 || a->attn.rel_pos) return fail(PA_ERR_BAD_SHAPE, "pa_p2t: attn.sr must be 1 (no reduction conv, no relative_pos)");
  if (a->n_levels < 1 || a->n_levels > 4) return fail(PA_ERR_BAD_SHAPE, "pa_p2t: n_levels must be 1..4");
  int M = 0;
  for (int l = 0; l < a->n_levels; ++l) {
    if (a->pool_h[l] < 1 || a->pool_w[l] < 1 || a->pool_h[l] > a->attn.Himg || a->pool_w[l] > a->attn.Wimg)
      return fail(PA_ERR_BAD_SHAPE, "pa_p2t: pooled size %dx%d of level %d must lie in [1, H] x [1, W]", a->pool_h[l], a->pool_w[l], l);
    M += a->pool_h[l] * a->pool_w[l];
  }
  *M_out = M;
  return PA_OK;
}

static pa_pvt_args p2t_attn_args(const pa_p2t_args* a, int M, const void* tokens) {
  pa_pvt_args at = a->attn;
  at.kv_tokens = tokens ? tokens : reinterpret_cast<const void*>(16);     // workspace sizing only needs it non-NULL
  at.kv_count = M;
  return at;
}

size_t pa_p2t_workspace_bytes(const pa_p2t_args* a) {
  int M = 0;
  if (p2t_check(a, &M)) return 0;
  const pa_pvt_args at = p2t_attn_args(a, M, nullptr);
  const size_t mrows = (size_t)a->attn.B * M;
  return align_up(mrows * a->attn.C * 4, 1024) + align_up(mrows * a->attn.C * 2, 1024) + pa_pvt_workspace_bytes(&at);
}

int pa_p2t_fwd(const pa_p2t_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int M = 0;
  int rc = p2t_check(a, &M);
  if (rc) return rc;
  if (!a->attn.x || !a->attn.q_weight || !a->attn.kv_weight || !a->attn.proj_weight || !a->attn.y || !a->norm_weight || !a->norm_bias)
    return fail(PA_ERR_NULL, "pa_p2t_fwd: x/weights/norm/y must be non-NULL");
  for (int l = 0; l < a->n_levels; ++l)
    if (!a->dconv_weight_t[l]) return fail(PA_ERR_NULL, "pa_p2t_fwd: dconv_weight_t[%d] is NULL", l);
  const size_t need = pa_p2t_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_p2t_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int C = a->attn.C;
  const long long mrows = (long long)a->attn.B * M;
  Arena ws(workspace);
  float* pooled = reinterpret_cast<float*>(ws.take((size_t)mrows * C * 4));
  void* tokens = ws.take((size_t)mrows * C * 2);
  P2tPoolParams pp = {};
  P2tTokParams tp = {};
  pp.x = a->attn.x; pp.pooled = pooled; pp.B = a->attn.B; pp.H = a->attn.Himg; pp.W = a->attn.Wimg; pp.C = C; pp.dtype = a->attn.dtype;
  pp.n_levels = a->n_levels; pp.M = M;
  tp.pooled = pooled; tp.out = tokens; tp.gamma = a->norm_weight; tp.beta = a->norm_bias; tp.eps = a->norm_eps;
  tp.B = a->attn.B; tp.C = C; tp.n_levels = a->n_levels; tp.M = M;
  int off = 0;
  for (int l = 0; l < a->n_levels; ++l) {
    pp.ph[l] = tp.ph[l] = a->pool_h[l]; pp.pw[l] = tp.pw[l] = a->pool_w[l]; pp.off[l] = tp.off[l] = off;
    tp.w[l] = a->dconv_weight_t[l]; tp.bias[l] = a->dconv_bias[l];
    off += a->pool_h[l] * a->pool_w[l];
  }
  // pooling pyramid -> normalised tokens   (p2t.py:78-86)
  p2t_pool_kernel<<<grid_for(mrows * (C / 8), 256), 256, 0, st>>>(pp);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  p2t_tokens_kernel<<<(int)((mrows * 32 + 255) / 256), 256, 0, st>>>(tp);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  const pa_pvt_args at = p2t_attn_args(a, M, tokens);
  return pvt_run(&at, at.x, at.dtype, nullptr, ws.take(0), st);     // q, kv, attention, proj   (p2t.py:76, 88-94)
}

// ================================================================ pvt.Block / segformer.Block / cmt.Block, attention half
size_t pa_pvt_block_attn_workspace_bytes(const pa_pvt_block_args* b) {
  if (!b || pvt_check_full(&b->attn)) return 0;
  return align_up((size_t)b->attn.B * b->attn.N * b->attn.C * 2, 1024) + pa_pvt_workspace_bytes(&b->attn);
}

int pa_pvt_block_attn_fwd(const pa_pvt_block_args* b, void* workspace, size_t workspace_bytes, void* stream) {
  if (!b) return fail(PA_ERR_NULL, "pa_pvt_block_attn_fwd: args is NULL");
  const pa_pvt_args* a = &b->attn;
  int rc = pvt_check_full(a);
  if (rc) return rc;
  if ((rc = pvt_ptr_check(a, "pa_pvt_block_attn_fwd"))) return rc;
  if (!b->ln_weight || !b->ln_bias) return fail(PA_ERR_NULL, "pa_pvt_block_attn_fwd: ln_weight/ln_bias must be non-NULL");
  const size_t need = pa_pvt_block_attn_workspace_bytes(b);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_pvt_block_attn_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)a->B * a->N;
  Arena ws(workspace);
  void* img = ws.take((size_t)rows * a->C * 2);
  // img = norm1(x)   (pvt.py:106, segformer.py:76, cmt.py:131), fp16
  LnParams ln;
  ln.x = a->x; ln.out = img; ln.gamma = b->ln_weight; ln.beta = b->ln_bias; ln.rows = rows; ln.C = a->C; ln.dtype = a->dtype; ln.eps = b->ln_eps;
  launch_layernorm(ln, st);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  // x + proj(attention(img)): the residual rides in the proj GEMM's epilogue
  return pvt_run(a, img, PA_DTYPE_F16, a->x, ws.take(0), st);
}

// ================================================================ CvT  (cvt.py:48-76)
static int cvt_check(const pa_cvt_args* a) {
  if (!a) return fail(PA_ERR_NULL, "pa_cvt: args is NULL");
  if (a->B <= 0 || a->C <= 0 || a->H <= 0 || a->Himg <= 0 || a->Wimg <= 0 || a->ks <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_cvt: sizes must be positive");
  if (a->C % a->H != 0) return fail(PA_ERR_BAD_SHAPE, "pa_cvt: dim %d not divisible by num_heads %d (cvt.py:51)", a->C, a->H);
  if (!attn_hd_ok(a->C / a->H)) return fail(PA_ERR_UNSUPPORTED, "pa_cvt: head_dim %d unsupported (multiples of 16 from 32 to 192)", a->C / a->H);
  if (a->dtype != PA_DTYPE_F16 && a->dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "pa_cvt: dtype must be fp16/bf16");
  return PA_OK;
}

size_t pa_cvt_workspace_bytes(const pa_cvt_args* a) {
  if (cvt_check(a)) return 0;
  const size_t rows = (size_t)a->B * a->Himg * a->Wimg;
  return align_up(rows * a->C * 2, 1024) * 2 + align_up(rows * 3 * a->C * 2, 1024) + 1024;
}

int pa_cvt_fwd(const pa_cvt_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = cvt_check(a);
  if (rc) return rc;
  if (!a->x || !a->dw_weight || !a->dw_scale || !a->dw_shift || !a->qkv_weight || !a->proj_weight || !a->y)
    return fail(PA_ERR_NULL, "pa_cvt_fwd: x/weights/y must be non-NULL");
  const size_t need = pa_cvt_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_cvt_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int C = a->C, HW = a->Himg * a->Wimg;
  const long long rows = (long long)a->B * HW;
  Arena ws(workspace);
  void* tok = ws.take((size_t)rows * C * 2);
  void* ob = ws.take((size_t)rows * C * 2);
  void* qkv = ws.take((size_t)rows * 3 * C * 2);
  // depthwise conv + eval BN, NCHW -> token-major   (cvt.py:55-57)
  DwParams dp;
  dp.x = a->x; dp.out = tok; dp.w = a->dw_weight; dp.scale = a->dw_scale; dp.shift = a->dw_shift;
  dp.B = a->B; dp.C = C; dp.H = a->Himg; dp.W = a->Wimg; dp.ks = a->ks; dp.dtype = a->dtype;
  const int dw3_smem = 32 * (((DW3_RB + 2) * a->Wimg) | 1) * (int)sizeof(float);
  if (a->ks == 3 && dw3_smem <= 48 * 1024 && a->B <= 65535) {
    dim3 grid(a->B, (C + 31) / 32, (a->Himg + DW3_RB - 1) / DW3_RB);
    dwconv3_bn_to_tokens_kernel<<<grid, 256, dw3_smem, st>>>(dp);
  } else {
    dim3 grid((HW + 31) / 32, (C + 31) / 32, a->B);
    dwconv_bn_to_tokens_kernel<<<grid, 256, 0, st>>>(dp);
  }
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  // 1x1 conv == linear over channels   (cvt.py:58), rows ordered (s,h,d) as ViT (cvt.py:66)
  if ((rc = linear(tok, PA_DTYPE_F16, C, a->qkv_weight, PA_DTYPE_F16, a->qkv_bias, qkv, PA_DTYPE_F16, 3 * C, rows, 3 * C, C, st))) return rc;
  AttnLaunch at = {};
  at.hd = C / a->H; at.G = a->B; at.H = a->H; at.n_q = HW; at.n_k = HW;
  at.q = qkv; at.ldq = 3 * C; at.q_group = (long long)HW * 3 * C; at.q_col0 = 0;
  at.k = qkv; at.v = qkv; at.ldk = 3 * C; at.k_group = (long long)HW * 3 * C; at.k_col0 = C; at.v_col0 = 2 * C;
  at.o = ob; at.ldo = C; at.o_group = (long long)HW * C; at.o_col0 = 0;
  at.scale = a->scale;
  if ((rc = attn_launch(at, st))) return rc;
  // proj 1x1 conv straight into NCHW: y[b] [C, HW] = Wp [C, C] . O[b]^T  + bias per row   (cvt.py:74)
  pa_gemm_args g = {};
  g.a_dtype = PA_DTYPE_F16; g.b_dtype = PA_DTYPE_F16; g.out_dtype = a->out_dtype;
  g.M = C; g.N = HW; g.K = C; g.Z = a->B;
  g.A = a->proj_weight; g.lda = C; g.a_batch = 0;
  g.B = ob; g.ldb = C; g.b_batch = (long long)HW * C;
  g.D = a->y; g.ldd = HW; g.d_batch = (long long)C * HW;
  g.bias = a->proj_bias; g.bias_mode = a->proj_bias ? 2 : 0;
  if (a->residual) { g.residual = a->residual; g.ldr = HW; g.r_batch = (long long)C * HW; g.res_dtype = a->dtype; }
  return gemm_impl(&g, st);
}

// ================================================================ XCiT  (xcit.py:233-265, 159-188)
static int xc_check(const pa_xcit_args* a, const char* who) {
  if (!a) return fail(PA_ERR_NULL, "%s: args is NULL", who);
  if (a->B <= 0 || a->N <= 0 || a->C <= 0 || a->H <= 0) return fail(PA_ERR_BAD_SHAPE, "%s: B,N,C,H must be positive", who);
  if (a->C % a->H != 0) return fail(PA_ERR_BAD_SHAPE, "%s: dim %d not divisible by num_heads %d", who, a->C, a->H);
  if (a->C / a->H != 64 && a->C / a->H != 32) return fail(PA_ERR_UNSUPPORTED, "%s: head_dim %d unsupported (64 or 32)", who, a->C / a->H);
  if (a->dtype != PA_DTYPE_F16 && a->dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "%s: dtype must be fp16/bf16", who);
  return PA_OK;
}

size_t pa_xca_workspace_bytes(const pa_xcit_args* a) {
  if (xc_check(a, "pa_xca")) return 0;
  const size_t rows = (size_t)a->B * a->N;
  return align_up(rows * 3 * a->C * 2, 1024) + align_up(rows * a->C * 2, 1024) + 1024;
}

// qkv GEMM -> cross-covariance core -> proj GEMM (+ residual).  x_in: the qkv GEMM's operand (a->x or the LayerNorm output).
static int xca_run(const pa_xcit_args* a, const void* x_in, int x_dtype, const void* residual, void* workspace, cudaStream_t st) {
  int rc;
  const int C = a->C;
  const long long rows = (long long)a->B * a->N;
  Arena ws(workspace);
  void* qkv = ws.take((size_t)rows * 3 * C * 2);
  void* ob = ws.take((size_t)rows * C * 2);
  if ((rc = linear(x_in, x_dtype, C, a->qkv_weight, x_dtype, a->qkv_bias, qkv, PA_DTYPE_F16, 3 * C, rows, 3 * C, C, st))) return rc;
  // cross-covariance core on the tensor cores (pa_xca.cuh): one unit per (image, 128-channel group)
  {
    CUtensorMap tm;
    uint64_t dims[3] = {(uint64_t)(3 * C), (uint64_t)a->N, (uint64_t)a->B};
    uint64_t str[2] = {(uint64_t)(3 * C) * 2, (uint64_t)a->N * 3 * C * 2};
    uint32_t box[3] = {64, 128, 1};
    if ((rc = make_tmap_16b(&tm, PA_DTYPE_F16, qkv, 3, dims, str, box, TM_SWZ_128))) return rc;
    XcaTcParams xp = {};
    xp.B = a->B; xp.N = a->N; xp.C = C; xp.H = a->H;
    xp.groups = (C + 127) / 128; xp.units = a->B * xp.groups; xp.nchunks = (a->N + 127) / 128;
    xp.temperature = a->temperature; xp.out = ob;
    xp.idesc_mn = make_idesc(128, 128, PA_F16, PA_F16, 1, 1);
    xp.idesc_k = make_idesc(128, 128, PA_F16, PA_F16, 0, 0);
    const int grid = xp.units < num_sms() ? xp.units : num_sms();
    if (C / a->H == 64) {
      static SmemAttr smem_attr;
      if ((rc = smem_attr.ensure(xca_tc_kernel<64>, XT_SMEM))) return rc;
      xca_tc_kernel<64><<<grid, XT_THREADS, XT_SMEM, st>>>(tm, xp);
    } else {
      static SmemAttr smem_attr;
      if ((rc = smem_attr.ensure(xca_tc_kernel<32>, XT_SMEM))) return rc;
      xca_tc_kernel<32><<<grid, XT_THREADS, XT_SMEM, st>>>(tm, xp);
    }
    PA_CUDA_OK(cudaGetLastError());
    launch_counter()++;
  }
  return linear(ob, PA_DTYPE_F16, C, a->proj_weight, PA_DTYPE_F16, a->proj_bias, a->y, a->out_dtype, C, rows, C, C, st,
                residual, C, a->dtype);
}

int pa_xca_fwd(const pa_xcit_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = xc_check(a, "pa_xca");
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->proj_weight || !a->temperature || !a->y) return fail(PA_ERR_NULL, "pa_xca_fwd: x/weights/temperature/y must be non-NULL");
  const size_t need = pa_xca_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_xca_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  return xca_run(a, a->x, a->dtype, nullptr, workspace, (cudaStream_t)stream);
}

// ---------------------------------------------------------------- xcit.XCABlock, attention half (xcit.py:291)
size_t pa_xca_block_attn_workspace_bytes(const pa_xca_block_args* b) {
  if (!b || xc_check(&b->attn, "pa_xca_block_attn")) return 0;
  return align_up((size_t)b->attn.B * b->attn.N * b->attn.C * 2, 1024) + pa_xca_workspace_bytes(&b->attn);
}

int pa_xca_block_attn_fwd(const pa_xca_block_args* b, void* workspace, size_t workspace_bytes, void* stream) {
  if (!b) return fail(PA_ERR_NULL, "pa_xca_block_attn_fwd: args is NULL");
  const pa_xcit_args* a = &b->attn;
  int rc = xc_check(a, "pa_xca_block_attn");
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->proj_weight || !a->temperature || !a->y || !b->ln_weight || !b->ln_bias)
    return fail(PA_ERR_NULL, "pa_xca_block_attn_fwd: x/weights/temperature/y/ln_weight/ln_bias must be non-NULL");
  if (a->C % 8) return fail(PA_ERR_BAD_SHAPE, "pa_xca_block_attn_fwd: dim must be a multiple of 8");
  const size_t need = pa_xca_block_attn_workspace_bytes(b);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_xca_block_attn_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)a->B * a->N;
  Arena ws(workspace);
  void* img = ws.take((size_t)rows * a->C * 2);
  LnParams ln;
  ln.x = a->x; ln.out = img; ln.gamma = b->ln_weight; ln.beta = b->ln_bias; ln.rows = rows; ln.C = a->C; ln.dtype = a->dtype; ln.eps = b->ln_eps;
  launch_layernorm(ln, st);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return xca_run(a, img, PA_DTYPE_F16, a->x, ws.take(0), st);
}

size_t pa_class_attn_workspace_bytes(const pa_xcit_args* a) {
  if (xc_check(a, "pa_class_attn")) return 0;
  const size_t rows = (size_t)a->B * a->N;
  return align_up(rows * 3 * a->C * 2, 1024) + align_up((size_t)a->B * a->C * 2, 1024) + 1024;
}

int pa_class_attn_fwd(const pa_xcit_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = xc_check(a, "pa_class_attn");
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->proj_weight || !a->y) return fail(PA_ERR_NULL, "pa_class_attn_fwd: x/weights/y must be non-NULL");
  if (a->out_dtype != a->dtype) return fail(PA_ERR_UNSUPPORTED, "pa_class_attn_fwd: y must have the dtype of x (patch tokens pass through unchanged, xcit.py:187)");
  const size_t need = pa_class_attn_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_class_attn_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int C = a->C;
  const long long rows = (long long)a->B * a->N;
  if (((long long)rows * C * 2) % 16) return fail(PA_ERR_MISALIGNED, "pa_class_attn_fwd: B*N*C must be a multiple of 8");
  Arena ws(workspace);
  void* qkv = ws.take((size_t)rows * 3 * C * 2);
  void* cls = ws.take((size_t)a->B * C * 2);
  if ((rc = linear(a->x, a->dtype, C, a->qkv_weight, a->dtype, a->qkv_bias, qkv, PA_DTYPE_F16, 3 * C, rows, 3 * C, C, st))) return rc;
  ClsParams cp;
  cp.qkv = qkv; cp.out = cls; cp.B = a->B; cp.N = a->N; cp.C = C; cp.H = a->H; cp.scale = a->scale;
  if (C / a->H == 64) class_attn_core_kernel<64><<<a->B * a->H, 256, a->N * sizeof(float), st>>>(cp);
  else class_attn_core_kernel<32><<<a->B * a->H, 256, a->N * sizeof(float), st>>>(cp);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  // y = x (patch tokens pass through, xcit.py:187), then row 0 of every image <- proj(cls)  (xcit.py:186)
  const long long n16 = rows * C * 2 / 16;
  copy16_kernel<<<grid_for(n16, 256), 256, 0, st>>>(reinterpret_cast<const uint4*>(a->x), reinterpret_cast<uint4*>(a->y), n16);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return linear(cls, PA_DTYPE_F16, C, a->proj_weight, PA_DTYPE_F16, a->proj_bias, a->y, a->out_dtype, (long long)a->N * C, a->B, C, C, st);
}

// ================================================================ CSWin  (cswin.py:51-127, 130-197)
static int lepe_geom(int resolution, int idx, int split, int* Hs, int* Ws) {
  if (idx == -1) { *Hs = resolution; *Ws = resolution; }
  else if (idx == 0) { *Hs = resolution; *Ws = split; }
  else if (idx == 1) { *Hs = split; *Ws = resolution; }
  else return fail(PA_ERR_UNSUPPORTED, "ERROR MODE %d (cswin.py:68-70: idx must be -1, 0 or 1)", idx);
  return PA_OK;
}

static int lepe_check(const pa_cswin_lepe_args* a) {
  if (!a) return fail(PA_ERR_NULL, "pa_cswin_lepe: args is NULL");
  if (a->B <= 0 || a->L <= 0 || a->C <= 0 || a->H <= 0 || a->resolution <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_cswin_lepe: sizes must be positive");
  if (a->L != a->resolution * a->resolution) return fail(PA_ERR_BAD_SHAPE, "flatten img_tokens has wrong size (cswin.py:110): L=%d, resolution=%d", a->L, a->resolution);
  if (a->C % a->H != 0) return fail(PA_ERR_BAD_SHAPE, "pa_cswin_lepe: dim %d not divisible by num_heads %d", a->C, a->H);
  if (a->C / a->H != 32 && a->C / a->H != 64) return fail(PA_ERR_UNSUPPORTED, "pa_cswin_lepe: head_dim %d unsupported (32 or 64)", a->C / a->H);
  int Hs, Ws;
  return lepe_geom(a->resolution, a->idx, a->split_size, &Hs, &Ws);
}

static int lepe_run(const pa_cswin_lepe_args* a, cudaStream_t st) {
  int Hs = 0, Ws = 0, rc;
  if ((rc = lepe_geom(a->resolution, a->idx, a->split_size, &Hs, &Ws))) return rc;
  if (a->resolution % Hs || a->resolution % Ws) return fail(PA_ERR_BAD_SHAPE, "pa_cswin_lepe: resolution %d not divisible by window %dx%d", a->resolution, Hs, Ws);
  if (a->C % 8 || a->ld % 8 || a->ldo % 8) return fail(PA_ERR_MISALIGNED, "pa_cswin_lepe: channel counts / pitches must be multiples of 8");
  if ((rc = current_device_check())) return rc;
  if (a->batch_stride != (long long)a->L * a->ld || a->out_batch_stride != (long long)a->L * a->ldo)
    return fail(PA_ERR_UNSUPPORTED, "pa_cswin_lepe: batch pitch must equal L * row pitch");
  AttnLaunch at = {};
  at.hd = a->C / a->H; at.windowed = true; at.H = a->H;
  at.q = a->q; at.k = a->k; at.v = a->v;
  at.ldq = a->ld; at.q_group = a->batch_stride; at.ldk = a->ld; at.k_group = a->batch_stride;
  at.q_col0 = 0; at.k_col0 = 0; at.v_col0 = 0;
  at.o = a->out; at.ldo = a->ldo; at.o_group = a->out_batch_stride; at.o_col0 = 0;
  at.scale = a->scale;
  at.B = a->B; at.R = a->resolution; at.H_sp = Hs; at.W_sp = Ws;
  // ---- one kernel: windowed attention with the LePE term computed in its epilogue from the resident V (cswin.py:116-125)
  if (!env().cswin_two_kernels) {
    AttnPlan plan;
    at.add_into_out = 0;
    if ((rc = attn_prepare(at, &plan))) return rc;
    rc = at.hd == 64 ? launch_attn_win<64>(plan, a, st) : launch_attn_win<32>(plan, a, st);
    if (rc <= 0) return rc;
  }
  // ---- fallback (window too large for the resident plan): LePE first, out = dwconv3x3(v) per window (cswin.py:93-96) ...
  LepeParams lp;
  lp.v = a->v; lp.out = a->out; lp.w = a->get_v_weight_t; lp.bias = a->get_v_bias;
  lp.ldv = a->ld; lp.ldo = a->ldo; lp.v_col0 = 0; lp.o_col0 = 0;
  lp.B = a->B; lp.R = a->resolution; lp.Cb = a->C; lp.H_sp = Hs; lp.W_sp = Ws;
  const int lepe_smem = (LEPE_RB + 2) * a->resolution * 128;
  if (a->C % 64 == 0 && lepe_smem <= 48 * 1024) {
    const int nblk = a->B * ((a->resolution + LEPE_RB - 1) / LEPE_RB) * (a->C / 64);
    lepe_tiled_kernel<<<nblk, 256, lepe_smem, st>>>(lp);
  } else {
    lepe_kernel<<<grid_for((long long)a->B * a->L * (a->C / 8), 256), 256, 0, st>>>(lp);
  }
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  // ... then the windowed attention adds softmax(q k^T scale) v on top (cswin.py:116-121) and scatters to image order (122-125)
  at.add_into_out = 1;
  return attn_launch(at, st);
}

int pa_cswin_lepe_fwd(const pa_cswin_lepe_args* a, void* stream) {
  int rc = lepe_check(a);
  if (rc) return rc;
  if (!a->q || !a->k || !a->v || !a->get_v_weight_t || !a->get_v_bias || !a->out) return fail(PA_ERR_NULL, "pa_cswin_lepe_fwd: q/k/v/get_v/out must be non-NULL");
  return lepe_run(a, (cudaStream_t)stream);
}

static int blk_check(const pa_cswin_block_args* a) {
  if (!a) return fail(PA_ERR_NULL, "pa_cswin_block: args is NULL");
  if (a->B <= 0 || a->C <= 0 || a->H <= 0 || a->reso <= 0 || a->split_size <= 0) return fail(PA_ERR_BAD_SHAPE, "pa_cswin_block: sizes must be positive");
  if (a->L != a->reso * a->reso) return fail(PA_ERR_BAD_SHAPE, "flatten img_tokens has wrong size (cswin.py:183): L=%d, reso=%d", a->L, a->reso);
  const int branches = a->last_stage ? 1 : 2;
  if (a->H % branches || a->C % (2 * branches)) return fail(PA_ERR_BAD_SHAPE, "pa_cswin_block: dim/heads not divisible by the branch count");
  const int hd = (a->C / branches) / (a->H / branches);
  if (hd != 32 && hd != 64) return fail(PA_ERR_UNSUPPORTED, "pa_cswin_block: head_dim %d unsupported (32 or 64)", hd);
  if (a->C % 8) return fail(PA_ERR_BAD_SHAPE, "pa_cswin_block: dim must be a multiple of 8");
  if (a->dtype != PA_DTYPE_F16 && a->dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "pa_cswin_block: dtype must be fp16/bf16");
  return PA_OK;
}

size_t pa_cswin_block_attn_workspace_bytes(const pa_cswin_block_args* a) {
  if (blk_check(a)) return 0;
  const size_t rows = (size_t)a->B * a->L;
  return align_up(rows * a->C * 2, 1024) * 2 + align_up(rows * 3 * a->C * 2, 1024) + 1024;
}

int pa_cswin_block_attn_fwd(const pa_cswin_block_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = blk_check(a);
  if (rc) return rc;
  if (!a->x || !a->norm1_weight || !a->norm1_bias || !a->qkv_weight || !a->proj_weight || !a->get_v_weight_t[0] || !a->get_v_bias[0] || !a->y)
    return fail(PA_ERR_NULL, "pa_cswin_block_attn_fwd: x/norm1/qkv/proj/get_v/y must be non-NULL");
  const int branches = a->last_stage ? 1 : 2;
  if (branches == 2 && (!a->get_v_weight_t[1] || !a->get_v_bias[1])) return fail(PA_ERR_NULL, "pa_cswin_block_attn_fwd: second branch get_v missing");
  const size_t need = pa_cswin_block_attn_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_cswin_block_attn_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const int C = a->C;
  const long long rows = (long long)a->B * a->L;
  Arena ws(workspace);
  void* img = ws.take((size_t)rows * C * 2);
  void* att = ws.take((size_t)rows * C * 2);
  void* qkv = ws.take((size_t)rows * 3 * C * 2);
  // img = norm1(x)   (cswin.py:184)
  LnParams ln;
  ln.x = a->x; ln.out = img; ln.gamma = a->norm1_weight; ln.beta = a->norm1_bias; ln.rows = rows; ln.C = C; ln.dtype = a->dtype; ln.eps = a->ln_eps;
  launch_layernorm(ln, st);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  // qkv = Linear(C, 3C)(img), column o -> (s, c) = (o / C, o % C)   (cswin.py:185)
  if ((rc = linear(img, PA_DTYPE_F16, C, a->qkv_weight, PA_DTYPE_F16, a->qkv_bias, qkv, PA_DTYPE_F16, 3 * C, rows, 3 * C, C, st))) return rc;
  // branches on channel halves (cswin.py:187-192); each writes its half of `att` (the torch.cat of :190)
  const int Cb = C / branches;
  for (int br = 0; br < branches; ++br) {
    pa_cswin_lepe_args l = {};
    l.B = a->B; l.L = a->L; l.C = Cb; l.H = a->H / branches;
    l.resolution = a->reso; l.idx = a->last_stage ? -1 : br; l.split_size = a->split_size;
    l.scale = a->scale;
    const uint16_t* base = reinterpret_cast<const uint16_t*>(qkv) + br * Cb;
    l.q = base; l.k = base + C; l.v = base + 2 * C;
    l.ld = 3 * C; l.batch_stride = (long long)a->L * 3 * C;
    l.get_v_weight_t = a->get_v_weight_t[br]; l.get_v_bias = a->get_v_bias[br];
    l.out = reinterpret_cast<uint16_t*>(att) + br * Cb; l.ldo = C; l.out_batch_stride = (long long)a->L * C;
    if ((rc = lepe_run(&l, st))) return rc;
  }
  // y = x + proj(att)   (cswin.py:193-194)
  return linear(att, PA_DTYPE_F16, C, a->proj_weight, PA_DTYPE_F16, a->proj_bias, a->y, a->out_dtype, C, rows, C, C, st,
                a->residual ? a->x : nullptr, C, a->dtype);
}

// ================================================================ DilateFormer multi-scale dilated attention  (dilateformer.py:41-134)
static int dilate_check(const pa_dilate_args* a, const char* who) {
  if (!a) return fail(PA_ERR_NULL, "%s: args is NULL", who);
  if (a->B <= 0 || a->Himg <= 0 || a->Wimg <= 0 || a->C <= 0 || a->H <= 0) return fail(PA_ERR_BAD_SHAPE, "%s: B,H,W,C,num_heads must be positive", who);
  if (a->B > 65535) return fail(PA_ERR_UNSUPPORTED, "%s: batch %d exceeds 65535 images per call", who, a->B);
  if (a->n_dilation < 1 || a->n_dilation > DL_MAX_GROUPS)
    return fail(PA_ERR_UNSUPPORTED, "%s: %d dilation groups (1 to %d supported)", who, a->n_dilation, DL_MAX_GROUPS);
  if (a->H % a->n_dilation)
    return fail(PA_ERR_BAD_SHAPE, "%s: num_heads%d must be the times of num_dilation%d (dilateformer.py:77)", who, a->H, a->n_dilation);
  if (a->C % a->H) return fail(PA_ERR_BAD_SHAPE, "%s: dim %d not divisible by num_heads %d", who, a->C, a->H);
  if (a->kernel_size < 1 || a->kernel_size % 2 == 0)
    return fail(PA_ERR_BAD_SHAPE, "%s: kernel_size %d must be odd (an even kernel's unfold output does not reshape, dilateformer.py:55)", who, a->kernel_size);
  if (a->kernel_size > 7) return fail(PA_ERR_UNSUPPORTED, "%s: kernel_size %d unsupported (odd, up to 7)", who, a->kernel_size);
  for (int g = 0; g < a->n_dilation; ++g)
    if (a->dilation[g] < 1) return fail(PA_ERR_BAD_SHAPE, "%s: dilation[%d] = %d must be >= 1", who, g, a->dilation[g]);
  const int hd = a->C / a->H;
  if (hd % 8 || hd > 64) return fail(PA_ERR_UNSUPPORTED, "%s: head_dim %d unsupported (multiples of 8 up to 64)", who, hd);
  if (!(a->scale > 0.f)) return fail(PA_ERR_UNSUPPORTED, "%s: scale must be > 0", who);
  if (a->dtype != PA_DTYPE_F16 && a->dtype != PA_DTYPE_BF16) return fail(PA_ERR_UNSUPPORTED, "%s: dtype must be fp16/bf16", who);
  if (a->out_dtype < PA_DTYPE_F16 || a->out_dtype > PA_DTYPE_F32) return fail(PA_ERR_UNSUPPORTED, "%s: bad out_dtype", who);
  return PA_OK;
}

// Band height and shared memory of the dilated-attention kernel: 8 image rows per CTA, halved until the widest group's staged
// rows (at most kernel_size * band rows, whatever the dilation) fit 113 KB; when a single band row does not fit 227 KB the map
// is too wide for this group width: 4 * Wimg * pitch * min(Himg, 1 + dil*(k-1), k) bytes must fit (pa_b200.h).
static int dilate_plan(const pa_dilate_args* a, DilateParams* p, int* smem) {
  const int Cg = a->C / a->n_dilation;
  p->Cg = Cg;
  p->heads_g = a->H / a->n_dilation;
  p->pstride = (Cg / 8) % 2 ? Cg : Cg + 8;
  const int dmax = a->Himg > a->Wimg ? a->Himg : a->Wimg;
  for (int g = 0; g < a->n_dilation; ++g)   // a dilation >= max(H, W) puts every tap but the centre outside the map: same result
    p->dil[g] = a->dilation[g] < dmax ? a->dilation[g] : dmax;
  auto rows_for = [&](int rows) {
    int r = 0;
    for (int g = 0; g < a->n_dilation; ++g) {
      const int rg = dilate_staged_rows(rows, a->kernel_size, p->dil[g], a->Himg);
      r = rg > r ? rg : r;
    }
    return r;
  };
  auto bytes = [&](int rows) { return 2ll * rows_for(rows) * a->Wimg * p->pstride * 2; };
  int rows = a->Himg < 8 ? a->Himg : 8;
  while (rows > 1 && bytes(rows) > 113 * 1024) rows /= 2;
  if (bytes(rows) > 227 * 1024)
    return fail(PA_ERR_UNSUPPORTED, "pa_dilate: %d staged rows of %d pixels x %d channels exceed shared memory (map too wide)",
                rows_for(rows), a->Wimg, Cg);
  p->rows = rows;
  *smem = (int)bytes(rows);
  return PA_OK;
}

extern "C++" template <int HD>
int launch_dilate_t(const DilateParams& p, int smem, int ng, cudaStream_t st) {
  static SmemAttr attr;
  int rc = attr.ensure(dilate_attn_kernel<HD>, smem);
  if (rc) return rc;
  dim3 grid((p.Himg + p.rows - 1) / p.rows, ng, p.B);
  dilate_attn_kernel<HD><<<grid, DL_THREADS, smem, st>>>(p);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  return PA_OK;
}

// O[B*H*W, C] = dilated attention of qkv[B*H*W, 3C] (both fp16, 16-byte aligned); arguments already checked by dilate_check.
// Plans (shared memory) and checks the device before the launch.
static int dilate_launch(const pa_dilate_args* a, const void* qkv, void* o, cudaStream_t st) {
  if ((reinterpret_cast<uintptr_t>(qkv) & 15) || (reinterpret_cast<uintptr_t>(o) & 15))
    return fail(PA_ERR_MISALIGNED, "pa_dilate: qkv / O buffers must be 16-byte aligned");
  DilateParams p = {};
  int smem = 0, rc;
  if ((rc = dilate_plan(a, &p, &smem))) return rc;
  if ((rc = current_device_check())) return rc;
  p.qkv = reinterpret_cast<const uint16_t*>(qkv);
  p.o = reinterpret_cast<uint16_t*>(o);
  p.B = a->B; p.Himg = a->Himg; p.Wimg = a->Wimg; p.C = a->C; p.ks = a->kernel_size;
  p.scale_log2 = a->scale * 1.4426950408889634f;
  switch (a->C / a->H) {
    case 8:  return launch_dilate_t<8>(p, smem, a->n_dilation, st);
    case 16: return launch_dilate_t<16>(p, smem, a->n_dilation, st);
    case 24: return launch_dilate_t<24>(p, smem, a->n_dilation, st);
    case 32: return launch_dilate_t<32>(p, smem, a->n_dilation, st);
    case 40: return launch_dilate_t<40>(p, smem, a->n_dilation, st);
    case 48: return launch_dilate_t<48>(p, smem, a->n_dilation, st);
    case 56: return launch_dilate_t<56>(p, smem, a->n_dilation, st);
    case 64: return launch_dilate_t<64>(p, smem, a->n_dilation, st);
    default: return fail(PA_ERR_UNSUPPORTED, "pa_dilate: head_dim %d unsupported", a->C / a->H);
  }
}

int pa_dilate_core(const pa_dilate_args* a, const void* qkv, void* o, void* stream) {
  int rc = dilate_check(a, "pa_dilate_core");
  if (rc) return rc;
  if (!qkv || !o) return fail(PA_ERR_NULL, "pa_dilate_core: qkv/o must be non-NULL");
  return dilate_launch(a, qkv, o, (cudaStream_t)stream);
}

size_t pa_dilate_workspace_bytes(const pa_dilate_args* a) {
  if (dilate_check(a, "pa_dilate")) return 0;
  const size_t rows = (size_t)a->B * a->Himg * a->Wimg;
  return align_up(rows * 3 * a->C * 2, 1024) + align_up(rows * a->C * 2, 1024) + 1024;
}

// qkv GEMM -> dilated attention -> proj GEMM (+ residual in its epilogue).  x_in: the qkv GEMM's A operand (a->x, or the
// LayerNorm output of the block entry point); residual: nullptr or the block input (dtype a->dtype, pitch C).
static int dilate_run(const pa_dilate_args* a, const void* x_in, int x_dtype, const void* residual, Arena& ws, cudaStream_t st) {
  int rc;
  const int C = a->C;
  const long long rows = (long long)a->B * a->Himg * a->Wimg;
  void* qkv = ws.take((size_t)rows * 3 * C * 2);
  void* obuf = ws.take((size_t)rows * C * 2);
  // qkv = 1x1 conv (dilateformer.py:88) on channels-last tokens: a token-major GEMM with the [3C, C] weight
  if ((rc = linear(x_in, x_dtype, C, a->qkv_weight, x_dtype, a->qkv_bias, qkv, PA_DTYPE_F16, 3 * C, rows, 3 * C, C, st))) return rc;
  if ((rc = dilate_launch(a, qkv, obuf, st))) return rc;
  // y = proj(O) (+ x)   (dilateformer.py:95, 130)
  return linear(obuf, PA_DTYPE_F16, C, a->proj_weight, PA_DTYPE_F16, a->proj_bias, a->y, a->out_dtype, C, rows, C, C, st,
                residual, C, a->dtype);
}

int pa_dilate_fwd(const pa_dilate_args* a, void* workspace, size_t workspace_bytes, void* stream) {
  int rc = dilate_check(a, "pa_dilate_fwd");
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->proj_weight || !a->y) return fail(PA_ERR_NULL, "pa_dilate_fwd: x/qkv_weight/proj_weight/y must be non-NULL");
  DilateParams p = {};
  int smem = 0;
  if ((rc = dilate_plan(a, &p, &smem))) return rc;
  const size_t need = pa_dilate_workspace_bytes(a);
  if (!workspace || workspace_bytes < need) return fail(PA_ERR_WORKSPACE, "pa_dilate_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  Arena ws(workspace);
  return dilate_run(a, a->x, a->dtype, nullptr, ws, (cudaStream_t)stream);
}

size_t pa_dilate_block_attn_workspace_bytes(const pa_dilate_block_args* b) {
  if (!b || dilate_check(&b->attn, "pa_dilate_block")) return 0;
  const size_t rows = (size_t)b->attn.B * b->attn.Himg * b->attn.Wimg;
  return align_up(rows * b->attn.C * 2, 1024) + pa_dilate_workspace_bytes(&b->attn);
}

int pa_dilate_block_attn_fwd(const pa_dilate_block_args* b, void* workspace, size_t workspace_bytes, void* stream) {
  if (!b) return fail(PA_ERR_NULL, "pa_dilate_block_attn_fwd: args is NULL");
  const pa_dilate_args* a = &b->attn;
  int rc = dilate_check(a, "pa_dilate_block_attn_fwd");
  if (rc) return rc;
  if (!a->x || !a->qkv_weight || !a->proj_weight || !a->y || !b->ln_weight || !b->ln_bias)
    return fail(PA_ERR_NULL, "pa_dilate_block_attn_fwd: x/qkv_weight/proj_weight/y/ln_weight/ln_bias must be non-NULL");
  DilateParams p = {};
  int smem = 0;
  if ((rc = dilate_plan(a, &p, &smem))) return rc;
  const size_t need = pa_dilate_block_attn_workspace_bytes(b);
  if (!workspace || workspace_bytes < need)
    return fail(PA_ERR_WORKSPACE, "pa_dilate_block_attn_fwd: workspace %zu B < required %zu B", workspace_bytes, need);
  if ((rc = current_device_check())) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const long long rows = (long long)a->B * a->Himg * a->Wimg;
  Arena ws(workspace);
  void* img = ws.take((size_t)rows * a->C * 2);
  // img = norm1(x)   (dilateformer.py:130), fp16
  LnParams ln;
  ln.x = a->x; ln.out = img; ln.gamma = b->ln_weight; ln.beta = b->ln_bias; ln.rows = rows; ln.C = a->C; ln.dtype = a->dtype; ln.eps = b->ln_eps;
  launch_layernorm(ln, st);
  PA_CUDA_OK(cudaGetLastError());
  launch_counter()++;
  // x + proj(attention(img)): the residual rides in the proj GEMM's epilogue
  return dilate_run(a, img, PA_DTYPE_F16, a->x, ws, st);
}

}  // extern "C"
