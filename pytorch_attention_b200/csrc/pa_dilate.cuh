// pa_dilate.cuh — multi-scale dilated attention core of DilateFormer (dilateformer.py:41-97, MultiDilatelocalAttention).
//
// qkv is the token-major output of the 1x1 qkv conv, [B*H*W, 3C] fp16 with column s*C + g*Cg + h*hd + d (part s, dilation
// group g, head h inside the group, channel d; dilateformer.py:88).  Query (y, x) of group g attends to the k*k keys at
// (y + i*dil_g - p, x + j*dil_g - p), p = dil_g*(k-1)/2, in row-major (i, j) order (nn.Unfold, dilateformer.py:48-60).  Unfold
// pads with zeros, so a key outside the map is a zero vector: its logit is exactly 0 and it stays in the softmax with a zero
// value.  O[token, g*Cg + h*hd + d] (dilateformer.py:90-94) is the K-major A operand of the proj GEMM.
//
// About 4*k*k*hd FLOP per (token, head) against 8 bytes per token and channel: HBM / L2 bound, no tensor cores.  One CTA per
// (band of R image rows, dilation group, image) stages the K and V rows its taps reach in shared memory once (cp.async,
// 16-byte chunks, all in flight before one wait), whole image rows at a time.  A small dilation stages one contiguous range,
// the band plus the p-row halo on both sides; once that range is longer than k*R rows (dilation > R) it stages k separate
// R-row slots instead, one per tap row i at y0 + i*dil - p, so shared memory never exceeds k*R rows whatever the dilation.
// Rows and columns outside the map are not staged: the kernel knows they are zero.  Each thread owns one (pixel, head): q is read once from global memory, the
// logits are computed twice from shared memory (max pass, then exp / sum / accumulate pass) so that no k*k-sized array is
// needed in registers, and O is written with 16-byte stores.
#pragma once
#include "pa_ptx.cuh"

namespace pa {

constexpr int DL_THREADS = 256;
constexpr int DL_MAX_GROUPS = 8;

struct DilateParams {
  const uint16_t* qkv;       // [B*H*W, 3C] fp16
  uint16_t* o;               // [B*H*W, C] fp16
  int B, Himg, Wimg, C, Cg, heads_g, ks;
  int rows;                  // image rows per CTA (band height)
  int pstride;               // staged pixel pitch in halves (Cg, padded to an odd number of 16-byte chunks)
  int dil[DL_MAX_GROUPS];
  float scale_log2;          // scale * log2(e)
};

// Staging of a band of `rows` rows for a group of dilation `dil`: one contiguous range (the band plus its halo, clipped to the
// map) while that is no longer than ks separate per-tap-row slots of `rows` rows each, else those slots.
__host__ __device__ inline bool dilate_contiguous(int rows, int ks, int dil, int Himg) {
  long long r = rows + (long long)dil * (ks - 1);
  if (r > Himg) r = Himg;
  return r <= (long long)ks * rows;
}
__host__ __device__ inline int dilate_staged_rows(int rows, int ks, int dil, int Himg) {
  if (!dilate_contiguous(rows, ks, dil, Himg)) return ks * rows;
  const long long r = rows + (long long)dil * (ks - 1);
  return r < Himg ? (int)r : Himg;
}

__device__ __forceinline__ void cp_async16(void* smem, const void* gmem) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(smem)), "l"(gmem) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

template <int HD>
__device__ __forceinline__ float dl_dot(const float (&q)[HD], const uint16_t* k) {
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < HD / 8; ++c) {
    const uint4 u = *reinterpret_cast<const uint4*>(k + 8 * c);
    const __half2* h = reinterpret_cast<const __half2*>(&u);
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 f = __half22float2(h[e]);
      s = fmaf(q[8 * c + 2 * e], f.x, s);
      s = fmaf(q[8 * c + 2 * e + 1], f.y, s);
    }
  }
  return s;
}

// One CTA's work; CONTIG selects the staging (contiguous range or per-tap-row slots), so each path compiles on its own.
template <int HD, bool CONTIG>
__device__ __forceinline__ void dilate_attn_cta(const DilateParams& p, uint16_t* dl_smem, int dil) {
  const int band = blockIdx.x, g = blockIdx.y, b = blockIdx.z;
  const int Himg = p.Himg, Wimg = p.Wimg, C = p.C, Cg = p.Cg, ks = p.ks;
  const int pad = dil * (ks - 1) / 2;
  const int R = p.rows;
  const int y0 = band * R;
  constexpr bool contig = CONTIG;
  const int ys0 = max(y0 - pad, 0);                                     // first staged image row (contiguous staging)
  const int n_rows = contig ? min(y0 + R - 1 + pad, Himg - 1) - ys0 + 1 : ks * R;
  const long long ld = 3ll * C;
  const long long img0 = (long long)b * Himg * Wimg;
  uint16_t* ks_ = dl_smem;                                              // K: [n_rows][Wimg][pstride]
  uint16_t* vs_ = dl_smem + (size_t)dilate_staged_rows(R, ks, dil, Himg) * Wimg * p.pstride;   // V, same layout

  // ---- stage K and V of the rows the band's taps reach, channels of group g.  Staged row s holds image row ys0 + s
  // (contiguous) or y0 + i*dil - pad + r with s = i*R + r (per tap row; rows outside the map or below the band are skipped).
  {
    const int chunks = Cg / 8;
    const int per_row = Wimg * chunks;
    const int total = n_rows * per_row;
    const uint16_t* kbase = p.qkv + img0 * ld + C + g * Cg;
    for (int t = threadIdx.x; t < total; t += DL_THREADS) {
      const int pix = t / chunks, c = t - pix * chunks;                  // pix = s * Wimg + x
      int gpix = ys0 * Wimg + pix;                                       // contiguous: staged row s is image row ys0 + s
      if (!contig) {
        const int s = pix / Wimg, x = pix - s * Wimg;
        const int i = s / R, r = s - i * R;
        const int yy = y0 + i * dil - pad + r;
        if (yy < 0 || yy >= Himg || y0 + r >= Himg) continue;
        gpix = yy * Wimg + x;
      }
      const uint16_t* src = kbase + (long long)gpix * ld + 8 * c;
      const int dst = pix * p.pstride + 8 * c;
      cp_async16(ks_ + dst, src);
      cp_async16(vs_ + dst, src + C);
    }
    cp_async_wait_all();
    __syncthreads();
  }

  // ---- one (pixel, head) per thread; consecutive threads take consecutive pixels of one head (conflict-free: odd pitch)
  const int band_px = R * Wimg;
  const int items = band_px * p.heads_g;
  for (int it = threadIdx.x; it < items; it += DL_THREADS) {
    const int h = it / band_px;
    const int pix = it - h * band_px;
    const int ry = pix / Wimg, x = pix - ry * Wimg;
    const int y = y0 + ry;
    if (y >= Himg) continue;
    const long long tok = img0 + (long long)y * Wimg + x;
    const int col = g * Cg + h * HD;
    float q[HD];
    {
      const uint16_t* qp = p.qkv + tok * ld + col;
#pragma unroll
      for (int c = 0; c < HD / 8; ++c) {
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(qp + 8 * c));
        const __half2* hh = reinterpret_cast<const __half2*>(&u);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float2 f = __half22float2(hh[e]);
          q[8 * c + 2 * e] = f.x * p.scale_log2;
          q[8 * c + 2 * e + 1] = f.y * p.scale_log2;
        }
      }
    }
    const uint16_t* kh = ks_ + h * HD;
    const uint16_t* vh = vs_ + h * HD;
    // pass 1: the row maximum of the k*k logits (log2 domain); a padded key's logit is 0
    float m = -INFINITY;
    for (int i = 0; i < ks; ++i) {
      const int yy = y + i * dil - pad;
      const bool row_in = yy >= 0 && yy < Himg;
      const int srow = contig ? yy - ys0 : i * R + ry;                 // staged row of tap row i
      for (int j = 0; j < ks; ++j) {
        const int xx = x + j * dil - pad;
        float s = 0.f;
        if (row_in && xx >= 0 && xx < Wimg) s = dl_dot<HD>(q, kh + (srow * Wimg + xx) * p.pstride);
        m = fmaxf(m, s);
      }
    }
    // pass 2: exponentials, their sum, and the weighted sum of the values (a padded key adds to the sum only)
    float acc[HD];
#pragma unroll
    for (int d = 0; d < HD; ++d) acc[d] = 0.f;
    float l = 0.f;
    for (int i = 0; i < ks; ++i) {
      const int yy = y + i * dil - pad;
      const bool row_in = yy >= 0 && yy < Himg;
      const int srow = contig ? yy - ys0 : i * R + ry;
      for (int j = 0; j < ks; ++j) {
        const int xx = x + j * dil - pad;
        if (row_in && xx >= 0 && xx < Wimg) {
          const int off = (srow * Wimg + xx) * p.pstride;
          const float e = ex2f(dl_dot<HD>(q, kh + off) - m);
          l += e;
          const uint16_t* vp = vh + off;
#pragma unroll
          for (int c = 0; c < HD / 8; ++c) {
            const uint4 u = *reinterpret_cast<const uint4*>(vp + 8 * c);
            const __half2* hh = reinterpret_cast<const __half2*>(&u);
#pragma unroll
            for (int k2 = 0; k2 < 4; ++k2) {
              const float2 f = __half22float2(hh[k2]);
              acc[8 * c + 2 * k2] = fmaf(e, f.x, acc[8 * c + 2 * k2]);
              acc[8 * c + 2 * k2 + 1] = fmaf(e, f.y, acc[8 * c + 2 * k2 + 1]);
            }
          }
        } else {
          l += ex2f(-m);
        }
      }
    }
    const float inv = 1.f / l;
    uint4* op = reinterpret_cast<uint4*>(p.o + tok * C + col);
#pragma unroll
    for (int c = 0; c < HD / 8; ++c) {
      uint4 u;
      u.x = pack_h2(acc[8 * c + 0] * inv, acc[8 * c + 1] * inv);
      u.y = pack_h2(acc[8 * c + 2] * inv, acc[8 * c + 3] * inv);
      u.z = pack_h2(acc[8 * c + 4] * inv, acc[8 * c + 5] * inv);
      u.w = pack_h2(acc[8 * c + 6] * inv, acc[8 * c + 7] * inv);
      op[c] = u;
    }
  }
}

template <int HD>
__global__ void __launch_bounds__(DL_THREADS) dilate_attn_kernel(const __grid_constant__ DilateParams p) {
  extern __shared__ __align__(16) uint16_t dl_smem[];
  int dil = 1;
#pragma unroll
  for (int i = 0; i < DL_MAX_GROUPS; ++i)                             // constant indices: the parameter array stays in param space
    if (i == (int)blockIdx.y) dil = p.dil[i];
  if (dilate_contiguous(p.rows, p.ks, dil, p.Himg)) dilate_attn_cta<HD, true>(p, dl_smem, dil);
  else dilate_attn_cta<HD, false>(p, dl_smem, dil);
}

}  // namespace pa
