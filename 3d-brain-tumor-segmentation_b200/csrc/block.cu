// b3d — ResnetBlock epilogue (reference layers/resnet.py:121-137), fused:
//   chse = sigmoid(relu(mean_vox(res) W1) W2)                         (tiny 1-CTA kernel)
//   out  = res * (sigmoid(res . w_sp) + chse) + relu(GN2(h2))         (one pass: 2 reads + 1 write)
// and its backward as two passes (reductions, then elementwise), SURVEY App. D.
// HBM-bound; T = F/4 lanes cooperate on one voxel (128-bit loads, shuffle reduce of the
// per-voxel channel dot).  GN2 follows the contiguous-chunk semantics of norm.cu and requires
// voxel-aligned chunks (D*H*W % groups == 0); otherwise callers use HAS_GN=0 + the norm.cu kernels.
#include "common.cuh"
#include "twin16.cuh"

namespace b3d {

constexpr int kBT = 256;
constexpr int kMaxNPL = 4;

struct BlockGeom {
  long long S;        // voxels per sample
  long long vpc;      // voxels per chunk (S / G)
  int F, T, npl;      // channels, lanes per voxel, float4 per lane
  int G, cg;
  int vox_per_cta;    // voxels handled by one CTA
  // depth-slab form (forward twin kernel only; batch 1): the tensors hold voxels [vshift, vshift + S_local) of the
  // volume S / vpc describe.  S_local < 0: the tensors are the volume
  long long vshift, S_local;
  int chunk0;         // first chunk the grid covers (slab form: only the chunks that intersect the slab are launched)
};

__device__ __forceinline__ float group_sum(float v, int T) {
  for (int o = T >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

__device__ __forceinline__ void moments(const double* __restrict__ stats, int chunk, double inv_L, float eps,
                                        float& mean, float& rstd) {
  const double s0 = stats[2 * chunk], s1 = stats[2 * chunk + 1];
  const double m = s0 * inv_L;
  double var = s1 * inv_L - m * m;
  var = var < 0.0 ? 0.0 : var;
  mean = (float)m;
  rstd = (float)(1.0 / sqrt(var + (double)eps));
}

// grid: (segments per chunk, B*G).  Each CTA walks vox_per_cta voxels of one chunk.
template <bool HAS_GN, int NPL>
__global__ void __launch_bounds__(kBT)
    block_epilogue_fwd_kernel(const float* __restrict__ res, const float* __restrict__ h2,
                              const double* __restrict__ stats, const float* __restrict__ gamma,
                              const float* __restrict__ beta, const float* __restrict__ wsp,
                              const float* __restrict__ chse, float* __restrict__ out, BlockGeom gm, float eps) {
  const int chunk = blockIdx.y, b = chunk / gm.G, g = chunk % gm.G;
  const int T = gm.T, lane = threadIdx.x % T, vl = threadIdx.x / T, vstep = kBT / T;
  float mean = 0.f, rstd = 1.f;
  if (HAS_GN) moments(stats, chunk, 1.0 / ((double)gm.vpc * gm.F), eps, mean, rstd);
  float4 w4[NPL], c4[NPL], ga4[NPL], be4[NPL];
#pragma unroll
  for (int q = 0; q < NPL; ++q)
    {
      const int c = (q * T + lane) * 4;
      w4[q] = *reinterpret_cast<const float4*>(wsp + c);
      c4[q] = *reinterpret_cast<const float4*>(chse + (long long)b * gm.F + c);
      if (HAS_GN) {
        float ga[4], be[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int j = g * gm.cg + (c + i) % gm.cg;
          ga[i] = gamma[j];
          be[i] = beta[j];
        }
        ga4[q] = make_float4(ga[0], ga[1], ga[2], ga[3]);
        be4[q] = make_float4(be[0], be[1], be[2], be[3]);
      }
    }
  const long long v0 = (long long)blockIdx.x * gm.vox_per_cta;
  const long long vend = min(v0 + gm.vox_per_cta, gm.vpc);
  const long long vbase = ((long long)b * gm.S + (long long)g * gm.vpc);
  const int iters = (int)((vend - v0 + vstep - 1) / vstep);   // CTA-uniform: whole warps stay in the shuffles
  for (int it = 0; it < iters; ++it) {
    const long long v = v0 + (long long)it * vstep + vl;
    const bool act = v < vend;
    const long long eo = (vbase + (act ? v : v0)) * gm.F;
    float4 r[NPL], h[NPL];
    float dot = 0.f;
#pragma unroll
    for (int q = 0; q < NPL; ++q)
      {
        const int c = (q * T + lane) * 4;
        r[q] = ld_stream(reinterpret_cast<const float4*>(res + eo + c));
        h[q] = ld_stream(reinterpret_cast<const float4*>(h2 + eo + c));
        dot += r[q].x * w4[q].x + r[q].y * w4[q].y + r[q].z * w4[q].z + r[q].w * w4[q].w;
      }
    dot = group_sum(dot, T);
    const float s = sigmoidf_(dot);
    if (act) {
#pragma unroll
      for (int q = 0; q < NPL; ++q)
        {
          const int c = (q * T + lane) * 4;
          float4 a = h[q];
          if (HAS_GN) {
            a.x = fmaxf((a.x - mean) * rstd * ga4[q].x + be4[q].x, 0.f);
            a.y = fmaxf((a.y - mean) * rstd * ga4[q].y + be4[q].y, 0.f);
            a.z = fmaxf((a.z - mean) * rstd * ga4[q].z + be4[q].z, 0.f);
            a.w = fmaxf((a.w - mean) * rstd * ga4[q].w + be4[q].w, 0.f);
          }
          float4 o;
          o.x = r[q].x * (s + c4[q].x) + a.x;
          o.y = r[q].y * (s + c4[q].y) + a.y;
          o.z = r[q].z * (s + c4[q].z) + a.z;
          o.w = r[q].w * (s + c4[q].w) + a.w;
          st_stream(reinterpret_cast<float4*>(out + eo + c), o);
        }
    }
  }
}

// Backward pass A — reductions.  Accumulates (atomics; outputs pre-zeroed by the host wrapper):
//   dchse[b][c] += sum_v do*res ; dwsp[c] += sum_v dlogit*res ; dgamma_j, dbeta_j ; csum[chunk] = (S1,S2)
template <bool HAS_GN, int NPL>
__global__ void __launch_bounds__(kBT)
    block_epilogue_bwd_reduce_kernel(const float* __restrict__ dout, const float* __restrict__ res,
                                     const float* __restrict__ h2, const double* __restrict__ stats,
                                     const float* __restrict__ gamma, const float* __restrict__ beta,
                                     const float* __restrict__ wsp, float* __restrict__ dchse,
                                     float* __restrict__ dwsp, float* __restrict__ dgamma,
                                     float* __restrict__ dbeta, double* __restrict__ csum, BlockGeom gm, float eps) {
  extern __shared__ float sm[];  // [4][F]: dchse, dwsp, dgam(c), dbet(c)
  for (int i = threadIdx.x; i < 4 * gm.F; i += kBT) sm[i] = 0.f;
  __syncthreads();
  const int chunk = blockIdx.y, b = chunk / gm.G, g = chunk % gm.G;
  const int T = gm.T, lane = threadIdx.x % T, vl = threadIdx.x / T, vstep = kBT / T;
  float mean = 0.f, rstd = 1.f;
  if (HAS_GN) moments(stats, chunk, 1.0 / ((double)gm.vpc * gm.F), eps, mean, rstd);
  float4 w4[NPL], ga4[NPL], be4[NPL];
  float acc_c[NPL][4], acc_w[NPL][4], acc_g[NPL][4], acc_b[NPL][4];
#pragma unroll
  for (int q = 0; q < NPL; ++q) {
#pragma unroll
    for (int i = 0; i < 4; ++i) acc_c[q][i] = acc_w[q][i] = acc_g[q][i] = acc_b[q][i] = 0.f;
    {
      const int c = (q * T + lane) * 4;
      w4[q] = *reinterpret_cast<const float4*>(wsp + c);
      if (HAS_GN) {
        float ga[4], be[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int j = g * gm.cg + (c + i) % gm.cg;
          ga[i] = gamma[j];
          be[i] = beta[j];
        }
        ga4[q] = make_float4(ga[0], ga[1], ga[2], ga[3]);
        be4[q] = make_float4(be[0], be[1], be[2], be[3]);
      }
    }
  }
  float s1 = 0.f, s2 = 0.f;
  const long long v0 = (long long)blockIdx.x * gm.vox_per_cta;
  const long long vend = min(v0 + gm.vox_per_cta, gm.vpc);
  const long long vbase = ((long long)b * gm.S + (long long)g * gm.vpc);
  const int iters = (int)((vend - v0 + vstep - 1) / vstep);   // CTA-uniform: whole warps stay in the shuffles
  for (int it = 0; it < iters; ++it) {
    const long long v = v0 + (long long)it * vstep + vl;
    const bool act = v < vend;
    const long long eo = (vbase + (act ? v : v0)) * gm.F;
    float4 r[NPL], d[NPL];
    float dot = 0.f, ds = 0.f;
#pragma unroll
    for (int q = 0; q < NPL; ++q)
      {
        const int c = (q * T + lane) * 4;
        r[q] = ld_stream(reinterpret_cast<const float4*>(res + eo + c));
        d[q] = ld_stream(reinterpret_cast<const float4*>(dout + eo + c));
        if (!act) d[q] = make_float4(0.f, 0.f, 0.f, 0.f);
        dot += r[q].x * w4[q].x + r[q].y * w4[q].y + r[q].z * w4[q].z + r[q].w * w4[q].w;
        ds += r[q].x * d[q].x + r[q].y * d[q].y + r[q].z * d[q].z + r[q].w * d[q].w;
      }
    dot = group_sum(dot, T);
    ds = group_sum(ds, T);
    const float s = sigmoidf_(dot);
    const float dl = ds * s * (1.f - s);
#pragma unroll
    for (int q = 0; q < NPL; ++q)
      {
        const float rr[4] = {r[q].x, r[q].y, r[q].z, r[q].w};
        const float dd[4] = {d[q].x, d[q].y, d[q].z, d[q].w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          acc_c[q][i] += dd[i] * rr[i];
          acc_w[q][i] += dl * rr[i];
        }
        if (HAS_GN) {
          const int c = (q * T + lane) * 4;
          const float4 hv = ld_stream(reinterpret_cast<const float4*>(h2 + eo + c));
          const float hh[4] = {hv.x, hv.y, hv.z, hv.w};
          const float ga[4] = {ga4[q].x, ga4[q].y, ga4[q].z, ga4[q].w};
          const float be[4] = {be4[q].x, be4[q].y, be4[q].z, be4[q].w};
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const float xh = (hh[i] - mean) * rstd;
            const float gq = (xh * ga[i] + be[i]) > 0.f ? dd[i] : 0.f;
            acc_g[q][i] += gq * xh;
            acc_b[q][i] += gq;
            const float hq = gq * ga[i];
            s1 += hq;
            s2 += hq * xh;
          }
        }
      }
  }
  // lanes of a warp with equal (lane % T) hold the same channels: butterfly over the voxel sub-index first, so that
  // only T lanes per warp touch shared memory
  const int wl = threadIdx.x & 31;
#pragma unroll
  for (int q = 0; q < NPL; ++q) {
    const int c = (q * T + lane) * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float a0 = acc_c[q][i], a1 = acc_w[q][i], a2 = acc_g[q][i], a3 = acc_b[q][i];
      for (int o = 16; o >= T; o >>= 1) {
        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
        if (HAS_GN) {
          a2 += __shfl_xor_sync(0xffffffffu, a2, o);
          a3 += __shfl_xor_sync(0xffffffffu, a3, o);
        }
      }
      if (wl < T) {
        atomicAdd(&sm[0 * gm.F + c + i], a0);
        atomicAdd(&sm[1 * gm.F + c + i], a1);
        if (HAS_GN) {
          atomicAdd(&sm[2 * gm.F + c + i], a2);
          atomicAdd(&sm[3 * gm.F + c + i], a3);
        }
      }
    }
  }
  __shared__ double red[64];
  double dd2[2] = {(double)s1, (double)s2};
  block_sum<2, double>(dd2, red);
  if (HAS_GN && threadIdx.x == 0) {
    atomicAdd(&csum[2 * chunk], dd2[0]);
    atomicAdd(&csum[2 * chunk + 1], dd2[1]);
  }
  for (int c = threadIdx.x; c < gm.F; c += kBT) {
    atomicAdd(&dchse[(long long)b * gm.F + c], sm[c]);
    atomicAdd(&dwsp[c], sm[gm.F + c]);
    if (HAS_GN) {
      const int j = g * gm.cg + c % gm.cg;
      atomicAdd(&dgamma[j], sm[2 * gm.F + c]);
      atomicAdd(&dbeta[j], sm[3 * gm.F + c]);
    }
  }
}

// Backward pass B — elementwise:  dres, dh2
template <bool HAS_GN, int NPL>
__global__ void __launch_bounds__(kBT)
    block_epilogue_bwd_apply_kernel(const float* __restrict__ dout, const float* __restrict__ res,
                                    const float* __restrict__ h2, const double* __restrict__ stats,
                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                    const float* __restrict__ wsp, const float* __restrict__ chse,
                                    const float* __restrict__ dgap, const double* __restrict__ csum,
                                    float* __restrict__ dres, float* __restrict__ dh2, BlockGeom gm, float eps) {
  const int chunk = blockIdx.y, b = chunk / gm.G, g = chunk % gm.G;
  const int T = gm.T, lane = threadIdx.x % T, vl = threadIdx.x / T, vstep = kBT / T;
  float mean = 0.f, rstd = 1.f, m1 = 0.f, m2 = 0.f;
  if (HAS_GN) {
    const double L = (double)gm.vpc * gm.F;
    moments(stats, chunk, 1.0 / L, eps, mean, rstd);
    m1 = (float)(csum[2 * chunk] / L);
    m2 = (float)(csum[2 * chunk + 1] / L);
  }
  float4 w4[NPL], c4[NPL], g4[NPL], ga4[NPL], be4[NPL];
#pragma unroll
  for (int q = 0; q < NPL; ++q)
    {
      const int c = (q * T + lane) * 4;
      w4[q] = *reinterpret_cast<const float4*>(wsp + c);
      c4[q] = *reinterpret_cast<const float4*>(chse + (long long)b * gm.F + c);
      g4[q] = *reinterpret_cast<const float4*>(dgap + (long long)b * gm.F + c);
      if (HAS_GN) {
        float ga[4], be[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int j = g * gm.cg + (c + i) % gm.cg;
          ga[i] = gamma[j];
          be[i] = beta[j];
        }
        ga4[q] = make_float4(ga[0], ga[1], ga[2], ga[3]);
        be4[q] = make_float4(be[0], be[1], be[2], be[3]);
      }
    }
  const long long v0 = (long long)blockIdx.x * gm.vox_per_cta;
  const long long vend = min(v0 + gm.vox_per_cta, gm.vpc);
  const long long vbase = ((long long)b * gm.S + (long long)g * gm.vpc);
  const int iters = (int)((vend - v0 + vstep - 1) / vstep);   // CTA-uniform: whole warps stay in the shuffles
  for (int it = 0; it < iters; ++it) {
    const long long v = v0 + (long long)it * vstep + vl;
    const bool act = v < vend;
    const long long eo = (vbase + (act ? v : v0)) * gm.F;
    float4 r[NPL], d[NPL];
    float dot = 0.f, ds = 0.f;
#pragma unroll
    for (int q = 0; q < NPL; ++q)
      {
        const int c = (q * T + lane) * 4;
        r[q] = ld_stream(reinterpret_cast<const float4*>(res + eo + c));
        d[q] = ld_stream(reinterpret_cast<const float4*>(dout + eo + c));
        dot += r[q].x * w4[q].x + r[q].y * w4[q].y + r[q].z * w4[q].z + r[q].w * w4[q].w;
        ds += r[q].x * d[q].x + r[q].y * d[q].y + r[q].z * d[q].z + r[q].w * d[q].w;
      }
    dot = group_sum(dot, T);
    ds = group_sum(ds, T);
    const float s = sigmoidf_(dot);
    const float dl = ds * s * (1.f - s);
    if (act) {
#pragma unroll
      for (int q = 0; q < NPL; ++q)
        {
          const int c = (q * T + lane) * 4;
          float4 o;
          o.x = d[q].x * (s + c4[q].x) + dl * w4[q].x + g4[q].x;
          o.y = d[q].y * (s + c4[q].y) + dl * w4[q].y + g4[q].y;
          o.z = d[q].z * (s + c4[q].z) + dl * w4[q].z + g4[q].z;
          o.w = d[q].w * (s + c4[q].w) + dl * w4[q].w + g4[q].w;
          st_stream(reinterpret_cast<float4*>(dres + eo + c), o);
          if (HAS_GN) {
            const float4 hv = ld_stream(reinterpret_cast<const float4*>(h2 + eo + c));
            const float hh[4] = {hv.x, hv.y, hv.z, hv.w};
            const float dd[4] = {d[q].x, d[q].y, d[q].z, d[q].w};
            const float ga[4] = {ga4[q].x, ga4[q].y, ga4[q].z, ga4[q].w};
            const float be[4] = {be4[q].x, be4[q].y, be4[q].z, be4[q].w};
            float oo[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float xh = (hh[i] - mean) * rstd;
              const float gq = (xh * ga[i] + be[i]) > 0.f ? dd[i] : 0.f;
              oo[i] = rstd * (gq * ga[i] - m1 - xh * m2);
            }
            st_stream(reinterpret_cast<float4*>(dh2 + eo + c), make_float4(oo[0], oo[1], oo[2], oo[3]));
          }
        }
    }
  }
}

// ================================================================================================ P16 twin forms
// The same forward / backward-apply passes writing the 16-bit operand twins of their results ([B, D, H, C/8, W, 8],
// common.cuh) for the tcgen05 convs that consume them.  Lane mapping: T = F/8 lanes cooperate on one voxel and every
// lane owns ONE 16-byte cell (8 consecutive channels): two 128-bit loads per input tensor, one 128-bit store per twin
// (Twin16 and the 16-bit packing: twin16.cuh).
struct VoxPos { unsigned row, w; };
__device__ __forceinline__ VoxPos vox_pos(unsigned W, unsigned vox) {
  VoxPos k;
  k.row = vox / W;
  k.w = vox - k.row * W;
  return k;
}
__device__ __forceinline__ void vox_advance(unsigned W, VoxPos& k, unsigned dv) {
  k.w += dv;
  while (k.w >= W) { k.w -= W; ++k.row; }
}
__device__ __forceinline__ void cell_store(const Twin16& o, unsigned b, const VoxPos& k, unsigned c8, const float (&v)[8]) {
  if (o.p == nullptr) return;
  const unsigned long long idx = (((unsigned long long)b * o.rows + k.row) * o.C8 + c8) * o.W + k.w;
  o.p[idx] = make_uint4(pk16(v[0], v[1], o.bf16), pk16(v[2], v[3], o.bf16), pk16(v[4], v[5], o.bf16),
                        pk16(v[6], v[7], o.bf16));
  if (o.p2 != nullptr)
    o.p2[idx] = make_uint4(pk16(v[0], v[1], 1), pk16(v[2], v[3], 1), pk16(v[4], v[5], 1), pk16(v[6], v[7], 1));
}
// grid: (segments per chunk, B*G); gm.T = F/8 lanes per voxel
template <bool HAS_GN>
__global__ void __launch_bounds__(kBT)
    block_fwd16_kernel(const float* __restrict__ res, const float* __restrict__ h2, const double* __restrict__ stats,
                       const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ wsp,
                       const float* __restrict__ chse, float* __restrict__ out, BlockGeom gm, float eps, Twin16 tw) {
  pdl_trigger();
  pdl_wait();
  const int chunk = blockIdx.y + gm.chunk0, b = chunk / gm.G, g = chunk % gm.G;
  const int T = gm.T, lane = threadIdx.x % T, vl = threadIdx.x / T, vstep = kBT / T;
  const int c = lane * 8;
  float mean = 0.f, rstd = 1.f;
  if (HAS_GN) moments(stats, chunk, 1.0 / ((double)gm.vpc * gm.F), eps, mean, rstd);
  float w8[8], c8v[8], ga8[8], be8[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    w8[i] = wsp[c + i];
    c8v[i] = chse[(long long)b * gm.F + c + i];
    const int j = g * gm.cg + (c + i) % gm.cg;
    ga8[i] = HAS_GN ? rstd * gamma[j] : 1.f;
    be8[i] = HAS_GN ? beta[j] : 0.f;
  }
  long long v_lo = 0, v_hi = gm.vpc, vshift = 0;
  if (gm.S_local >= 0) {                                       // the part of this chunk inside the slab
    vshift = gm.vshift;
    v_lo = max(0LL, vshift - (long long)g * gm.vpc);
    v_hi = min(gm.vpc, vshift + gm.S_local - (long long)g * gm.vpc);
  }
  const long long v0 = v_lo + (long long)blockIdx.x * gm.vox_per_cta;
  const long long vend = min(v0 + gm.vox_per_cta, v_hi);
  if (v0 >= vend) return;                                      // CTA-uniform
  const long long vbase = ((long long)b * gm.S + (long long)g * gm.vpc) - vshift;
  const int iters = (int)((vend - v0 + vstep - 1) / vstep);   // CTA-uniform: whole warps stay in the shuffles
  VoxPos pos = vox_pos(tw.W, (unsigned)((long long)g * gm.vpc + v0 + vl - vshift));
  for (int it = 0; it < iters; ++it) {
    const long long v = v0 + (long long)it * vstep + vl;
    const bool act = v < vend;
    const long long eo = (vbase + (act ? v : v0)) * gm.F + c;
    float r[8], h[8];
    ld8(res + eo, r);
    ld8(h2 + eo, h);
    float dot = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) dot += r[i] * w8[i];
    dot = group_sum(dot, T);
    const float s = sigmoidf_(dot);
    if (act) {
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float a = HAS_GN ? fmaxf(fmaf(h[i] - mean, ga8[i], be8[i]), 0.f) : h[i];
        o[i] = r[i] * (s + c8v[i]) + a;
      }
      if (out != nullptr) st8(out + eo, o);
      cell_store(tw, (unsigned)b, pos, (unsigned)lane, o);
    }
    vox_advance(tw.W, pos, (unsigned)vstep);
  }
}

// dres, dh2 as bf16 twins (+ optional fp32) and their column sums (bias gradients of the pointwise / second conv)
template <bool HAS_DB>
__global__ void __launch_bounds__(kBT)
    block_bwd_apply16_kernel(const float* __restrict__ dout, const float* __restrict__ res,
                             const float* __restrict__ h2, const double* __restrict__ stats,
                             const float* __restrict__ gamma, const float* __restrict__ beta,
                             const float* __restrict__ wsp, const float* __restrict__ chse,
                             const float* __restrict__ dgap, const double* __restrict__ csum,
                             float* __restrict__ dres, float* __restrict__ dh2, BlockGeom gm, float eps, Twin16 tr,
                             Twin16 th, float* __restrict__ dbias_res, float* __restrict__ dbias_h2) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sdb[];      // [2][F]
  if (HAS_DB) {
    for (int i = threadIdx.x; i < 2 * gm.F; i += kBT) sdb[i] = 0.f;
    __syncthreads();
  }
  const int chunk = blockIdx.y, b = chunk / gm.G, g = chunk % gm.G;
  const int T = gm.T, lane = threadIdx.x % T, vl = threadIdx.x / T, vstep = kBT / T;
  const int c = lane * 8;
  float mean, rstd;
  const double L = (double)gm.vpc * gm.F;
  moments(stats, chunk, 1.0 / L, eps, mean, rstd);
  const float m1 = (float)(csum[2 * chunk] / L), m2 = (float)(csum[2 * chunk + 1] / L);
  float w8[8], c8v[8], g8[8], ga8[8], be8[8], ar[HAS_DB ? 8 : 1], ah[HAS_DB ? 8 : 1];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    w8[i] = wsp[c + i];
    c8v[i] = chse[(long long)b * gm.F + c + i];
    g8[i] = dgap[(long long)b * gm.F + c + i];
    const int j = g * gm.cg + (c + i) % gm.cg;
    ga8[i] = gamma[j];
    be8[i] = beta[j];
    if (HAS_DB) ar[i] = ah[i] = 0.f;
  }
  const long long v0 = (long long)blockIdx.x * gm.vox_per_cta;
  const long long vend = min(v0 + gm.vox_per_cta, gm.vpc);
  const long long vbase = ((long long)b * gm.S + (long long)g * gm.vpc);
  const int iters = (int)((vend - v0 + vstep - 1) / vstep);
  VoxPos pos = vox_pos(tr.W, (unsigned)((long long)g * gm.vpc + v0 + vl));
  // two voxels per thread and step: all six 32-byte loads are issued before the first shuffle reduction
  for (int it = 0; it < iters; it += 2) {
    float r[2][8], d[2][8], h[2][8];
    bool act[2];
    long long eo[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const long long v = v0 + (long long)(it + u) * vstep + vl;
      act[u] = it + u < iters && v < vend;
      eo[u] = (vbase + (act[u] ? v : v0)) * gm.F + c;
      ld8(res + eo[u], r[u]);
      ld8(dout + eo[u], d[u]);
      ld8(h2 + eo[u], h[u]);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      if (u == 1 && it + 1 >= iters) break;          // CTA-uniform: whole warps stay in the shuffles
      float dot = 0.f, ds = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) { dot += r[u][i] * w8[i]; ds += r[u][i] * d[u][i]; }
      dot = group_sum(dot, T);
      ds = group_sum(ds, T);
      const float s = sigmoidf_(dot);
      const float dl = ds * s * (1.f - s);
      if (act[u]) {
        float o1[8], o2[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          o1[i] = d[u][i] * (s + c8v[i]) + dl * w8[i] + g8[i];
          const float xh = (h[u][i] - mean) * rstd;
          const float gq = (xh * ga8[i] + be8[i]) > 0.f ? d[u][i] : 0.f;
          o2[i] = rstd * (gq * ga8[i] - m1 - xh * m2);
          if (HAS_DB) { ar[i] += o1[i]; ah[i] += o2[i]; }
        }
        if (dres != nullptr) st8(dres + eo[u], o1);
        if (dh2 != nullptr) st8(dh2 + eo[u], o2);
        cell_store(tr, (unsigned)b, pos, (unsigned)lane, o1);
        cell_store(th, (unsigned)b, pos, (unsigned)lane, o2);
      }
      vox_advance(tr.W, pos, (unsigned)vstep);
    }
  }
  if (HAS_DB) {
    // lanes of a warp with equal (lane % T) hold the same channels: butterfly over the voxel sub-index first
    const int wl = threadIdx.x & 31;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float a0 = ar[i], a1 = ah[i];
      for (int o = 16; o >= T; o >>= 1) {
        a0 += __shfl_xor_sync(0xffffffffu, a0, o);
        a1 += __shfl_xor_sync(0xffffffffu, a1, o);
      }
      if (wl < T) {
        atomicAdd(&sdb[c + i], a0);
        atomicAdd(&sdb[gm.F + c + i], a1);
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < gm.F; i += kBT) {
      atomicAdd(&dbias_res[i], sdb[i]);
      atomicAdd(&dbias_h2[i], sdb[gm.F + i]);
    }
  }
}

// Backward pass A (reductions) in the cell-per-lane form: T = F/8 lanes per voxel, 8 consecutive channels per lane, all
// per-channel accumulators and constants in registers (the float4-per-lane form above keeps 16 partial sums per lane
// pair and runs at 60 % of the HBM peak at 128^3 x 16).
__global__ void __launch_bounds__(kBT)
    block_bwd_reduce8_kernel(const float* __restrict__ dout, const float* __restrict__ res,
                             const float* __restrict__ h2, const double* __restrict__ stats,
                             const float* __restrict__ gamma, const float* __restrict__ beta,
                             const float* __restrict__ wsp, float* __restrict__ dchse, float* __restrict__ dwsp,
                             float* __restrict__ dgamma, float* __restrict__ dbeta, double* __restrict__ csum,
                             BlockGeom gm, float eps) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];  // [4][F]: dchse, dwsp, dgam(c), dbet(c)
  for (int i = threadIdx.x; i < 4 * gm.F; i += kBT) sm[i] = 0.f;
  __syncthreads();
  const int chunk = blockIdx.y, b = chunk / gm.G, g = chunk % gm.G;
  const int T = gm.T, lane = threadIdx.x % T, vl = threadIdx.x / T, vstep = kBT / T;
  const int c = lane * 8;
  float mean, rstd;
  moments(stats, chunk, 1.0 / ((double)gm.vpc * gm.F), eps, mean, rstd);
  float w8[8], ga8[8], be8[8], ac[8], aw[8], ag[8], ab[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    w8[i] = wsp[c + i];
    const int j = g * gm.cg + (c + i) % gm.cg;
    ga8[i] = gamma[j];
    be8[i] = beta[j];
    ac[i] = aw[i] = ag[i] = ab[i] = 0.f;
  }
  float s1 = 0.f, s2 = 0.f;
  const long long v0 = (long long)blockIdx.x * gm.vox_per_cta;
  const long long vend = min(v0 + gm.vox_per_cta, gm.vpc);
  const long long vbase = ((long long)b * gm.S + (long long)g * gm.vpc);
  const int iters = (int)((vend - v0 + vstep - 1) / vstep);   // CTA-uniform: whole warps stay in the shuffles
  // two voxels per thread and step: all six 32-byte loads are issued before the first shuffle reduction
  for (int it = 0; it < iters; it += 2) {
    float r[2][8], d[2][8], h[2][8];
    bool act[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const long long v = v0 + (long long)(it + u) * vstep + vl;
      act[u] = it + u < iters && v < vend;
      const long long eo = (vbase + (act[u] ? v : v0)) * gm.F + c;
      ld8(res + eo, r[u]);
      ld8(dout + eo, d[u]);
      ld8(h2 + eo, h[u]);
    }
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      float dot = 0.f, ds = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        if (!act[u]) d[u][i] = 0.f;
        dot += r[u][i] * w8[i];
        ds += r[u][i] * d[u][i];
      }
      dot = group_sum(dot, T);
      ds = group_sum(ds, T);
      const float s = sigmoidf_(dot);
      const float dl = ds * s * (1.f - s);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        ac[i] += d[u][i] * r[u][i];
        aw[i] += dl * r[u][i];
        const float xh = (h[u][i] - mean) * rstd;
        const float gq = (xh * ga8[i] + be8[i]) > 0.f ? d[u][i] : 0.f;
        ag[i] += gq * xh;
        ab[i] += gq;
        const float hq = gq * ga8[i];
        s1 += hq;
        s2 += hq * xh;
      }
    }
  }
  // lanes of a warp with equal (lane % T) hold the same channels: butterfly over the voxel sub-index first
  const int wl = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float a0 = ac[i], a1 = aw[i], a2 = ag[i], a3 = ab[i];
    for (int o = 16; o >= T; o >>= 1) {
      a0 += __shfl_xor_sync(0xffffffffu, a0, o);
      a1 += __shfl_xor_sync(0xffffffffu, a1, o);
      a2 += __shfl_xor_sync(0xffffffffu, a2, o);
      a3 += __shfl_xor_sync(0xffffffffu, a3, o);
    }
    if (wl < T) {
      atomicAdd(&sm[0 * gm.F + c + i], a0);
      atomicAdd(&sm[1 * gm.F + c + i], a1);
      atomicAdd(&sm[2 * gm.F + c + i], a2);
      atomicAdd(&sm[3 * gm.F + c + i], a3);
    }
  }
  __shared__ double red[64];
  double dd2[2] = {(double)s1, (double)s2};
  block_sum<2, double>(dd2, red);
  if (threadIdx.x == 0) {
    atomicAdd(&csum[2 * chunk], dd2[0]);
    atomicAdd(&csum[2 * chunk + 1], dd2[1]);
  }
  for (int cc = threadIdx.x; cc < gm.F; cc += kBT) {
    atomicAdd(&dchse[(long long)b * gm.F + cc], sm[cc]);
    atomicAdd(&dwsp[cc], sm[gm.F + cc]);
    const int j = g * gm.cg + cc % gm.cg;
    atomicAdd(&dgamma[j], sm[2 * gm.F + cc]);
    atomicAdd(&dbeta[j], sm[3 * gm.F + cc]);
  }
}

// ---- channel squeeze-excitation FCs (resnet.py:121-124); one CTA, loops over the batch ----------
// The matrices are tiny (F x R, F <= 512) but the kernels sit on the critical path 32 times per training step, so what
// counts is the LENGTH of the dependent load chains: both products are split over all 256 threads.
//   colvec: out[n] = sum_m v[m] * W[m*N + n]  (n contiguous): thread (part, n) sums rows m = part (mod P), P = 256 / N
//           partial sums, combined through shared memory
//   rowvec: out[r] = sum_j W[r*L + j] * v[j]  (j contiguous): one warp per row, lanes over j, shuffle reduction
constexpr int kSeThreads = 256;
template <class Fin>
__device__ __forceinline__ void se_colvec(const float* __restrict__ v, const float* __restrict__ W, int M, int N,
                                          float* __restrict__ red, Fin finish) {
  int P = 1;
  while (P * 2 * N <= kSeThreads) P *= 2;
  for (int n0 = 0; n0 < N; n0 += kSeThreads) {          // N > 256: one pass per 256 outputs (P = 1)
    const int t = threadIdx.x, n = n0 + t % (N < kSeThreads ? N : kSeThreads), part = N < kSeThreads ? t / N : 0;
    float a = 0.f;
    if (part < P && n < N) {
#pragma unroll 8
      for (int m = part; m < M; m += P) a += v[m] * __ldg(W + (long long)m * N + n);
    }
    if (P > 1) {
      if (part < P) red[part * N + n] = a;
      __syncthreads();
      if (t < N) {
        a = red[t];
        for (int q = 1; q < P; ++q) a += red[q * N + t];
        finish(t, a);
      }
      __syncthreads();
    } else if (n < N) {
      finish(n, a);
    }
  }
}
template <class Fin>
__device__ __forceinline__ void se_rowvec(const float* __restrict__ W, const float* __restrict__ v, int Rows, int L,
                                          Fin finish) {
  // four rows per warp and step: their loads and shuffle reductions are independent and overlap
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int r0 = warp * 4; r0 < Rows; r0 += (kSeThreads / 32) * 4) {
    float a[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = lane; j < L; j += 32) {
      const float vj = v[j];
#pragma unroll
      for (int u = 0; u < 4; ++u)
        if (r0 + u < Rows) a[u] += __ldg(W + (long long)(r0 + u) * L + j) * vj;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) a[u] = warp_sum(a[u]);
#pragma unroll
    for (int u = 0; u < 4; ++u)
      if (lane == 0 && r0 + u < Rows) finish(r0 + u, a[u]);
  }
}

__global__ void __launch_bounds__(kSeThreads)
    se_fc_fwd_kernel(const float* __restrict__ gap_sum, const float* __restrict__ w1, const float* __restrict__ w2,
                     float* __restrict__ hidden, float* __restrict__ chse, int B, int F, int R, float inv_vox) {
  extern __shared__ float sm[];  // mean[F], hid[R], red[256]
  float* mean = sm;
  float* hid = sm + F;
  float* red = hid + R;
  for (int b = 0; b < B; ++b) {
    for (int c = threadIdx.x; c < F; c += kSeThreads) mean[c] = gap_sum[b * F + c] * inv_vox;
    __syncthreads();
    se_colvec(mean, w1, F, R, red, [&](int k, float a) {
      a = fmaxf(a, 0.f);
      hid[k] = a;
      hidden[b * R + k] = a;
    });
    __syncthreads();
    se_colvec(hid, w2, R, F, red, [&](int c, float a) { chse[b * F + c] = 1.f / (1.f + expf(-a)); });
    __syncthreads();
  }
}

__global__ void __launch_bounds__(kSeThreads)
    se_fc_bwd_kernel(const float* __restrict__ gap_sum, const float* __restrict__ w1, const float* __restrict__ w2,
                     const float* __restrict__ hidden, const float* __restrict__ chse,
                     const float* __restrict__ dchse, float* __restrict__ dw1, float* __restrict__ dw2,
                     float* __restrict__ dgap, int B, int F, int R, float inv_vox) {
  extern __shared__ float sm[];  // dz2[F], dz1[R], red[256]
  float* dz2 = sm;
  float* dz1 = sm + F;
  for (int b = 0; b < B; ++b) {
    for (int c = threadIdx.x; c < F; c += kSeThreads) {
      const float y = chse[b * F + c];
      dz2[c] = dchse[b * F + c] * y * (1.f - y);
    }
    __syncthreads();
    se_rowvec(w2, dz2, R, F, [&](int k, float a) { dz1[k] = hidden[b * R + k] > 0.f ? a : 0.f; });
    __syncthreads();
    for (int i = threadIdx.x; i < F * R; i += kSeThreads) {
      const int k2 = i / F, c2 = i % F;              // dw2[k][c]
      const float g2 = hidden[b * R + k2] * dz2[c2];
      const int c1 = i / R, k1 = i % R;              // dw1[c][k]
      const float g1 = gap_sum[b * F + c1] * inv_vox * dz1[k1];
      dw2[i] = b == 0 ? g2 : dw2[i] + g2;
      dw1[i] = b == 0 ? g1 : dw1[i] + g1;
    }
    se_rowvec(w1, dz1, F, R, [&](int c, float a) { dgap[b * F + c] = a * inv_vox; });
    __syncthreads();
  }
}

static int block_geom(const TView& res, int groups, bool has_gn, BlockGeom* gm, int* nchunks) {
  const int F = (int)res.shape[res.ndim - 1];
  const long long B = res.shape[0];
  const long long S = res.numel / B / F;
  B3D_REQUIRE(F % 4 == 0, B3D_ERR_UNSUPPORTED, "block epilogue: filters (%d) must be a multiple of 4", F);
  int G = has_gn ? groups : 1;
  if (has_gn) {
    B3D_REQUIRE(F >= groups && F % groups == 0, B3D_ERR_SHAPE,
                "Number of groups (%d) must be a multiple of the number of channels (%d).", groups, F);
    B3D_REQUIRE(S % groups == 0, B3D_ERR_UNSUPPORTED,
                "fused GN epilogue needs D*H*W (%lld) divisible by groups (%d)", (long long)S, groups);
  } else {
    // no chunk structure needed: split every sample into up to 8 pseudo-chunks for grid parallelism
    G = 1;
  }
  int q = F / 4, T = 1;
  while (T < 32 && q % (T * 2) == 0) T *= 2;
  B3D_REQUIRE(q / T <= kMaxNPL, B3D_ERR_UNSUPPORTED, "block epilogue: unsupported filter count %d", F);
  gm->S = S;
  gm->vshift = 0; gm->S_local = -1; gm->chunk0 = 0;
  gm->vpc = S / G;
  gm->F = F;
  gm->T = T;
  gm->npl = q / T;
  gm->G = G;
  gm->cg = has_gn ? F / groups : F;
  const int vstep = kBT / T;
  // ~8 voxel-iterations per thread-group, but enough CTAs to fill the machine
  // ~16 voxel-iterations per thread-group at least, and no more than ~4 waves of CTAs in total (the reducing
  // kernels end in a handful of atomics per CTA)
  long long vp = (long long)vstep * 4;
  const long long cap = (4LL * sm_count() + B * G - 1) / (B * G);
  const long long need = ((gm->vpc + cap - 1) / cap + vstep - 1) / vstep * vstep;
  if (need > vp) vp = need;
  gm->vox_per_cta = (int)vp;
  *nchunks = (int)(B * G);
  B3D_REQUIRE(*nchunks <= 65535, B3D_ERR_SHAPE, "batch*groups too large");
  return B3D_OK;
}

// geometry of the cell kernels: T = F/8 lanes per voxel (a power of two <= 32)
static int block_geom16(const TView& res, int groups, bool has_gn, BlockGeom* gm, int* nchunks) {
  B3D_REQUIRE(res.ndim == 5, B3D_ERR_SHAPE, "block epilogue (P16): res must be [B, D, H, W, F]");
  B3D_TRY(block_geom(res, groups, has_gn, gm, nchunks));
  const int T = gm->F / 8;
  B3D_REQUIRE(gm->F % 8 == 0 && T >= 1 && T <= 32 && (T & (T - 1)) == 0, B3D_ERR_UNSUPPORTED,
              "block epilogue (P16): filters must be 8 * 2^k <= 256 (got %d)", gm->F);
  B3D_REQUIRE(res.numel / res.shape[0] / gm->F < (1LL << 32), B3D_ERR_UNSUPPORTED, "block epilogue (P16): sample too large");
  gm->T = T; gm->npl = 2;
  const int vstep = kBT / T;
  long long vp = (long long)vstep * 2;     // >= 2 voxel steps per thread; small tensors get many short CTAs, not a 16-step latency chain
  const long long B = res.shape[0];
  const long long cap = (3LL * sm_count() + B * gm->G - 1) / (B * gm->G);
  const long long need = ((gm->vpc + cap - 1) / cap + vstep - 1) / vstep * vstep;
  if (need > vp) vp = need;
  gm->vox_per_cta = (int)vp;
  return B3D_OK;
}

static inline dim3 block_grid(const BlockGeom& gm, int nchunks) {
  return dim3((unsigned)((gm.vpc + gm.vox_per_cta - 1) / gm.vox_per_cta), (unsigned)nchunks, 1);
}

// instantiate on the exact number of float4 per lane (registers: the accumulator arrays are sized by it)
#define B3D_NPL(npl, launch)                   \
  do {                                         \
    switch (npl) {                             \
      case 1: { constexpr int kN = 1; launch; } break; \
      case 2: { constexpr int kN = 2; launch; } break; \
      case 3: { constexpr int kN = 3; launch; } break; \
      default: { constexpr int kN = 4; launch; } break; \
    }                                          \
  } while (0)

static int vecF(const DLTensor* t, long long n, const char* name, TView* v) {
  B3D_TRY(view(t, DT_F32, -1, false, name, v));
  B3D_REQUIRE(v->numel == n, B3D_ERR_SHAPE, "%s: expected %lld values, got %lld", name, n, (long long)v->numel);
  return B3D_OK;
}

}  // namespace b3d

using namespace b3d;

extern "C" int b3d_se_fc_fwd(const DLTensor* gap_sum_, const DLTensor* w1_, const DLTensor* w2_,
                             DLTensor* hidden_, DLTensor* chse_, float inv_vox, void* stream) {
  TView gs, w1, w2, hid, ch;
  B3D_TRY(view(gap_sum_, DT_F32, 2, false, "gap_sum", &gs));
  B3D_TRY(view(w1_, DT_F32, 2, false, "w1", &w1));
  B3D_TRY(view(w2_, DT_F32, 2, false, "w2", &w2));
  const int B = (int)gs.shape[0], F = (int)gs.shape[1], R = (int)w1.shape[1];
  B3D_REQUIRE(w1.shape[0] == F && w2.shape[0] == R && w2.shape[1] == F, B3D_ERR_SHAPE, "se_fc: weight shapes");
  B3D_TRY(vecF(hidden_, (long long)B * R, "hidden", &hid));
  B3D_TRY(vecF(chse_, (long long)B * F, "chse", &ch));
  se_fc_fwd_kernel<<<1, kSeThreads, sizeof(float) * (F + R + kSeThreads), (cudaStream_t)stream>>>(
      (const float*)gs.p, (const float*)w1.p, (const float*)w2.p, (float*)hid.p, (float*)ch.p, B, F, R, inv_vox);
  B3D_LAUNCH_CHECK("se_fc_fwd");
  return B3D_OK;
}

extern "C" int b3d_se_fc_bwd(const DLTensor* gap_sum_, const DLTensor* w1_, const DLTensor* w2_,
                             const DLTensor* hidden_, const DLTensor* chse_, const DLTensor* dchse_,
                             DLTensor* dw1_, DLTensor* dw2_, DLTensor* dgap_, float inv_vox, void* stream) {
  TView gs, w1, w2, hid, ch, dch, dw1, dw2, dg;
  B3D_TRY(view(gap_sum_, DT_F32, 2, false, "gap_sum", &gs));
  B3D_TRY(view(w1_, DT_F32, 2, false, "w1", &w1));
  B3D_TRY(view(w2_, DT_F32, 2, false, "w2", &w2));
  const int B = (int)gs.shape[0], F = (int)gs.shape[1], R = (int)w1.shape[1];
  B3D_REQUIRE(w1.shape[0] == F && w2.shape[0] == R && w2.shape[1] == F, B3D_ERR_SHAPE, "se_fc: weight shapes");
  B3D_TRY(vecF(hidden_, (long long)B * R, "hidden", &hid));
  B3D_TRY(vecF(chse_, (long long)B * F, "chse", &ch));
  B3D_TRY(vecF(dchse_, (long long)B * F, "dchse", &dch));
  B3D_TRY(vecF(dw1_, (long long)F * R, "dw1", &dw1));
  B3D_TRY(vecF(dw2_, (long long)F * R, "dw2", &dw2));
  B3D_TRY(vecF(dgap_, (long long)B * F, "dgap", &dg));
  se_fc_bwd_kernel<<<1, kSeThreads, sizeof(float) * (F + R + kSeThreads), (cudaStream_t)stream>>>(
      (const float*)gs.p, (const float*)w1.p, (const float*)w2.p, (const float*)hid.p, (const float*)ch.p,
      (const float*)dch.p, (float*)dw1.p, (float*)dw2.p, (float*)dg.p, B, F, R, inv_vox);
  B3D_LAUNCH_CHECK("se_fc_bwd");
  return B3D_OK;
}

// With the twin out16 (and out16b, a second, bf16 twin for the weight gradients of the consuming convs) given: the cell
// kernel, out nullable; otherwise the float4 kernel, out required.  total_vox != 0 (cell kernel only): res / h2 / the
// twin hold voxels [vox_offset, vox_offset + D*H*W) of a batch-1 volume of total_vox voxels (depth-slab inference);
// `stats` = the all-reduced GroupNorm statistics of the whole volume's chunks, `chse` from the all-reduced pooling sums.
extern "C" int b3d_block_epilogue_fwd(const DLTensor* res_, const DLTensor* h2_, const DLTensor* stats_,
                                      const DLTensor* gamma_, const DLTensor* beta_, const DLTensor* wsp_,
                                      const DLTensor* chse_, DLTensor* out_, DLTensor* out16_, DLTensor* out16b_,
                                      int groups, float eps, int has_gn, long long vox_offset, long long total_vox,
                                      void* stream) {
  B3D_REQUIRE(out16_ != nullptr || out16b_ == nullptr, B3D_ERR_ARG, "block epilogue: out16b without out16");
  TView res, h2, out, st, ga, be, wsp, ch;
  BlockGeom gm;
  int nchunks;
  B3D_TRY(view(res_, DT_F32, -1, false, "res", &res));
  B3D_TRY(view(h2_, DT_F32, -1, false, "h2", &h2));
  if (out_ != nullptr || out16_ == nullptr) B3D_TRY(view(out_, DT_F32, -1, false, "out", &out));
  B3D_REQUIRE(res.numel == h2.numel && (out_ == nullptr || res.numel == out.numel), B3D_ERR_SHAPE,
              "block epilogue: size mismatch");
  if (out16_ == nullptr) {
    B3D_REQUIRE(total_vox == 0, B3D_ERR_UNSUPPORTED, "block epilogue: a window needs the twin kernel");
    B3D_TRY(block_geom(res, groups, has_gn != 0, &gm, &nchunks));
  } else {
    B3D_REQUIRE(total_vox == 0 || (res.ndim == 5 && res.shape[0] == 1), B3D_ERR_SHAPE, "block epilogue (window): batch 1");
    B3D_TRY(block_geom16(res, groups, has_gn != 0, &gm, &nchunks));
  }
  int nlaunch = nchunks;
  if (total_vox != 0) {      // the window's CTAs keep their per-CTA voxel count, the grid covers the chunks it meets
    const long long S_local = gm.S;
    B3D_REQUIRE(total_vox > 0 && vox_offset >= 0 && vox_offset + S_local <= total_vox && total_vox % gm.G == 0 &&
                    total_vox < (1LL << 32), B3D_ERR_ARG, "block epilogue (window): bad window (%lld + %lld of %lld)",
                vox_offset, S_local, total_vox);
    gm.S = total_vox; gm.vpc = total_vox / gm.G; gm.vshift = vox_offset; gm.S_local = S_local;
    gm.chunk0 = (int)(vox_offset / gm.vpc);
    nlaunch = (int)((vox_offset + S_local - 1) / gm.vpc) - gm.chunk0 + 1;
  }
  B3D_TRY(vecF(wsp_, gm.F, "wsp", &wsp));
  B3D_TRY(vecF(chse_, res.shape[0] * gm.F, "chse", &ch));
  if (has_gn) {
    B3D_TRY(view(stats_, DT_F64, -1, false, "stats", &st));
    B3D_REQUIRE(st.numel == 2LL * nchunks, B3D_ERR_SHAPE, "stats: wrong size");
    B3D_TRY(vecF(gamma_, gm.F, "gamma", &ga));
    B3D_TRY(vecF(beta_, gm.F, "beta", &be));
  }
  cudaStream_t s = (cudaStream_t)stream;
  const dim3 grid = block_grid(gm, nlaunch);
  if (out16_ == nullptr) {
    if (has_gn) {
      B3D_NPL(gm.npl, (block_epilogue_fwd_kernel<true, kN><<<grid, kBT, 0, s>>>(
          (const float*)res.p, (const float*)h2.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p,
          (const float*)wsp.p, (const float*)ch.p, (float*)out.p, gm, eps)));
    } else {
      B3D_NPL(gm.npl, (block_epilogue_fwd_kernel<false, kN><<<grid, kBT, 0, s>>>(
          (const float*)res.p, (const float*)h2.p, nullptr, nullptr, nullptr, (const float*)wsp.p,
          (const float*)ch.p, (float*)out.p, gm, eps)));
    }
    B3D_LAUNCH_CHECK("block_epilogue_fwd");
    return B3D_OK;
  }
  Twin16 tw;
  B3D_TRY(twin_view(out16_, out16b_, res, &tw));
  if (has_gn)
    launch_pdl(block_fwd16_kernel<true>, grid, kBT, 0, s, (const float*)res.p, (const float*)h2.p, (const double*)st.p,
               (const float*)ga.p, (const float*)be.p, (const float*)wsp.p, (const float*)ch.p, (float*)out.p, gm, eps,
               tw);
  else
    launch_pdl(block_fwd16_kernel<false>, grid, kBT, 0, s, (const float*)res.p, (const float*)h2.p, nullptr, nullptr,
               nullptr, (const float*)wsp.p, (const float*)ch.p, (float*)out.p, gm, eps, tw);
  B3D_LAUNCH_CHECK("block_fwd16");
  return B3D_OK;
}

extern "C" int b3d_block_epilogue_bwd_reduce(const DLTensor* dout_, const DLTensor* res_, const DLTensor* h2_,
                                             const DLTensor* stats_, const DLTensor* gamma_,
                                             const DLTensor* beta_, const DLTensor* wsp_, DLTensor* dchse_,
                                             DLTensor* dwsp_, DLTensor* dgamma_, DLTensor* dbeta_,
                                             DLTensor* csum_, int groups, float eps, int has_gn, void* stream) {
  TView dout, res, h2, st, ga, be, wsp, dch, dws, dga, dbe, cs;
  BlockGeom gm;
  int nchunks;
  B3D_TRY(view(dout_, DT_F32, -1, false, "dout", &dout));
  B3D_TRY(view(res_, DT_F32, -1, false, "res", &res));
  B3D_REQUIRE(res.numel == dout.numel, B3D_ERR_SHAPE, "block epilogue bwd: size mismatch");
  B3D_TRY(block_geom(res, groups, has_gn != 0, &gm, &nchunks));
  B3D_TRY(vecF(wsp_, gm.F, "wsp", &wsp));
  B3D_TRY(vecF(dchse_, res.shape[0] * gm.F, "dchse", &dch));
  B3D_TRY(vecF(dwsp_, gm.F, "dwsp", &dws));
  cudaStream_t s = (cudaStream_t)stream;
  B3D_TRY(cuda_ok(cudaMemsetAsync(dch.p, 0, sizeof(float) * dch.numel, s), "memset"));
  B3D_TRY(cuda_ok(cudaMemsetAsync(dws.p, 0, sizeof(float) * gm.F, s), "memset"));
  const size_t smem = sizeof(float) * 4 * gm.F;
  if (has_gn) {
    B3D_TRY(view(h2_, DT_F32, -1, false, "h2", &h2));
    B3D_REQUIRE(res.numel == h2.numel, B3D_ERR_SHAPE, "block epilogue bwd: size mismatch");
    B3D_TRY(view(stats_, DT_F64, -1, false, "stats", &st));
    B3D_TRY(view(csum_, DT_F64, -1, false, "csum", &cs));
    B3D_REQUIRE(st.numel == 2LL * nchunks && cs.numel == 2LL * nchunks, B3D_ERR_SHAPE, "stats/csum: wrong size");
    B3D_TRY(vecF(gamma_, gm.F, "gamma", &ga));
    B3D_TRY(vecF(beta_, gm.F, "beta", &be));
    B3D_TRY(vecF(dgamma_, gm.F, "dgamma", &dga));
    B3D_TRY(vecF(dbeta_, gm.F, "dbeta", &dbe));
    B3D_TRY(cuda_ok(cudaMemsetAsync(cs.p, 0, sizeof(double) * 2 * nchunks, s), "memset"));
    B3D_TRY(cuda_ok(cudaMemsetAsync(dga.p, 0, sizeof(float) * gm.F, s), "memset"));
    B3D_TRY(cuda_ok(cudaMemsetAsync(dbe.p, 0, sizeof(float) * gm.F, s), "memset"));
    {
      const int T8 = gm.F / 8;
      if (res.ndim == 5 && gm.F % 8 == 0 && T8 >= 1 && T8 <= 32 && (T8 & (T8 - 1)) == 0) {
        BlockGeom g8 = gm;
        g8.T = T8; g8.npl = 2;
        const int vstep = kBT / T8;
        long long vp = (long long)vstep * 4;
        const long long Bn = res.shape[0];
        const long long cap = (3LL * sm_count() + Bn * gm.G - 1) / (Bn * gm.G);
        const long long need = ((gm.vpc + cap - 1) / cap + vstep - 1) / vstep * vstep;
        if (need > vp) vp = need;
        g8.vox_per_cta = (int)vp;
        launch_pdl(block_bwd_reduce8_kernel, block_grid(g8, nchunks), kBT, smem, s, (const float*)dout.p, (const float*)res.p, (const float*)h2.p, (const double*)st.p, (const float*)ga.p,
            (const float*)be.p, (const float*)wsp.p, (float*)dch.p, (float*)dws.p, (float*)dga.p, (float*)dbe.p,
            (double*)cs.p, g8, eps);
        B3D_LAUNCH_CHECK("block_bwd_reduce8");
        return B3D_OK;
      }
    }
    B3D_NPL(gm.npl, (block_epilogue_bwd_reduce_kernel<true, kN><<<block_grid(gm, nchunks), kBT, smem, s>>>(
        (const float*)dout.p, (const float*)res.p, (const float*)h2.p, (const double*)st.p, (const float*)ga.p,
        (const float*)be.p, (const float*)wsp.p, (float*)dch.p, (float*)dws.p, (float*)dga.p, (float*)dbe.p,
        (double*)cs.p, gm, eps)));
  } else {
    B3D_NPL(gm.npl, (block_epilogue_bwd_reduce_kernel<false, kN><<<block_grid(gm, nchunks), kBT, smem, s>>>(
        (const float*)dout.p, (const float*)res.p, nullptr, nullptr, nullptr, nullptr, (const float*)wsp.p,
        (float*)dch.p, (float*)dws.p, nullptr, nullptr, nullptr, gm, eps)));
  }
  B3D_LAUNCH_CHECK("block_epilogue_bwd_reduce");
  return B3D_OK;
}

// With a twin dres16 / dh216 given (bf16, for the data / weight gradients of the pointwise and the second 3x3x3 conv;
// fused-GroupNorm form only): the cell kernel; every gradient needs its fp32 output or its twin, and dbias_res /
// dbias_h2 (nullable, both or none) receive their column sums = those convs' bias gradients.  Otherwise the float4
// kernel: dres and, with has_gn, dh2 required.
extern "C" int b3d_block_epilogue_bwd_apply(const DLTensor* dout_, const DLTensor* res_, const DLTensor* h2_,
                                            const DLTensor* stats_, const DLTensor* gamma_,
                                            const DLTensor* beta_, const DLTensor* wsp_, const DLTensor* chse_,
                                            const DLTensor* dgap_, const DLTensor* csum_, DLTensor* dres_,
                                            DLTensor* dh2_, DLTensor* dres16_, DLTensor* dh216_,
                                            DLTensor* dbias_res_, DLTensor* dbias_h2_, int groups, float eps,
                                            int has_gn, void* stream) {
  const bool twins = dres16_ != nullptr || dh216_ != nullptr;
  B3D_REQUIRE((dres_ != nullptr || dres16_ != nullptr) && (!has_gn || dh2_ != nullptr || dh216_ != nullptr),
              B3D_ERR_ARG, "block epilogue bwd: every gradient needs an output");
  B3D_REQUIRE((dbias_res_ == nullptr) == (dbias_h2_ == nullptr), B3D_ERR_ARG,
              "block epilogue bwd: both bias gradients or none");
  B3D_REQUIRE(twins || dbias_res_ == nullptr, B3D_ERR_ARG, "block epilogue bwd: bias gradients without a twin");
  B3D_REQUIRE(!twins || has_gn, B3D_ERR_UNSUPPORTED, "block epilogue bwd (P16): the fused-GroupNorm form only");
  TView dout, res, h2, st, ga, be, wsp, ch, dg, cs, dres, dh2;
  BlockGeom gm;
  int nchunks;
  B3D_TRY(view(dout_, DT_F32, -1, false, "dout", &dout));
  B3D_TRY(view(res_, DT_F32, -1, false, "res", &res));
  if (dres_ != nullptr) B3D_TRY(view(dres_, DT_F32, -1, false, "dres", &dres));
  B3D_REQUIRE(res.numel == dout.numel && (dres_ == nullptr || res.numel == dres.numel), B3D_ERR_SHAPE,
              "block epilogue bwd: size mismatch");
  if (twins)
    B3D_TRY(block_geom16(res, groups, true, &gm, &nchunks));
  else
    B3D_TRY(block_geom(res, groups, has_gn != 0, &gm, &nchunks));
  B3D_TRY(vecF(wsp_, gm.F, "wsp", &wsp));
  B3D_TRY(vecF(chse_, res.shape[0] * gm.F, "chse", &ch));
  B3D_TRY(vecF(dgap_, res.shape[0] * gm.F, "dgap", &dg));
  if (has_gn) {
    B3D_TRY(view(h2_, DT_F32, -1, false, "h2", &h2));
    if (dh2_ != nullptr) B3D_TRY(view(dh2_, DT_F32, -1, false, "dh2", &dh2));
    B3D_REQUIRE(res.numel == h2.numel && (dh2_ == nullptr || res.numel == dh2.numel), B3D_ERR_SHAPE,
                "block epilogue bwd: size mismatch");
    B3D_TRY(view(stats_, DT_F64, -1, false, "stats", &st));
    B3D_TRY(view(csum_, DT_F64, -1, false, "csum", &cs));
    B3D_REQUIRE(st.numel == 2LL * nchunks && cs.numel == 2LL * nchunks, B3D_ERR_SHAPE, "stats/csum: wrong size");
    B3D_TRY(vecF(gamma_, gm.F, "gamma", &ga));
    B3D_TRY(vecF(beta_, gm.F, "beta", &be));
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (!twins) {
    if (has_gn) {
      B3D_NPL(gm.npl, (block_epilogue_bwd_apply_kernel<true, kN><<<block_grid(gm, nchunks), kBT, 0, s>>>(
          (const float*)dout.p, (const float*)res.p, (const float*)h2.p, (const double*)st.p, (const float*)ga.p,
          (const float*)be.p, (const float*)wsp.p, (const float*)ch.p, (const float*)dg.p, (const double*)cs.p,
          (float*)dres.p, (float*)dh2.p, gm, eps)));
    } else {
      B3D_NPL(gm.npl, (block_epilogue_bwd_apply_kernel<false, kN><<<block_grid(gm, nchunks), kBT, 0, s>>>(
          (const float*)dout.p, (const float*)res.p, nullptr, nullptr, nullptr, nullptr, (const float*)wsp.p,
          (const float*)ch.p, (const float*)dg.p, nullptr, (float*)dres.p, nullptr, gm, eps)));
    }
    B3D_LAUNCH_CHECK("block_epilogue_bwd_apply");
    return B3D_OK;
  }
  Twin16 tr, th;
  B3D_TRY(twin_view(dres16_, nullptr, res, &tr));
  B3D_TRY(twin_view(dh216_, nullptr, res, &th));
  float *dbr = nullptr, *dbh = nullptr;
  if (dbias_res_ != nullptr) {
    TView t;
    B3D_TRY(vecF(dbias_res_, gm.F, "dbias_res", &t));
    dbr = (float*)t.p;
    B3D_TRY(vecF(dbias_h2_, gm.F, "dbias_h2", &t));
    dbh = (float*)t.p;
    B3D_TRY(cuda_ok(cudaMemsetAsync(dbr, 0, sizeof(float) * gm.F, s), "memset"));
    B3D_TRY(cuda_ok(cudaMemsetAsync(dbh, 0, sizeof(float) * gm.F, s), "memset"));
  }
#define B3D_BWD16(DB)                                                                                              \
  launch_pdl(block_bwd_apply16_kernel<DB>, block_grid(gm, nchunks), kBT, DB ? sizeof(float) * 2 * gm.F : 0, s, \
      (const float*)dout.p, (const float*)res.p, (const float*)h2.p, (const double*)st.p, (const float*)ga.p,      \
      (const float*)be.p, (const float*)wsp.p, (const float*)ch.p, (const float*)dg.p, (const double*)cs.p,        \
      (float*)dres.p, (float*)dh2.p, gm, eps, tr, th, dbr, dbh)
  if (dbr != nullptr) B3D_BWD16(true); else B3D_BWD16(false);
#undef B3D_BWD16
  B3D_LAUNCH_CHECK("block_bwd_apply16");
  return B3D_OK;
}
