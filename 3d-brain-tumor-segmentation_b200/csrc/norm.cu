// b3d — GroupNormalization (reference layers/group_norm.py:83-124) in its channels_last form:
// "group" g of sample b is the g-th contiguous 1/G chunk of the sample's flat NDHWC buffer
// (SURVEY F1); the affine index of flat element e is  j = g*(C/G) + (e mod C) mod (C/G).
// HBM-bound: every kernel streams whole chunks with 128-bit accesses; reductions are
// per-thread fp32 -> warp shuffle -> block -> one fp64 atomic per CTA.
//
//   stats[b][g] = (sum x, sum x^2)  fp64   (also produced by the conv epilogues)
//   algorithmic bytes/elem: stats 4, apply 8, bwd_reduce 8, bwd_apply 12.
#include "common.cuh"
#include "twin16.cuh"

namespace b3d {

constexpr int kThreads = 256;
constexpr int kIter = 8;  // float4 per thread per CTA
constexpr int kIterR = 4; // ... in the two-operand reducing kernel (register budget)

struct ChunkGeom {
  long long L;     // elements per chunk
  int C, cg, G;    // channels, channels per group, groups
  float inv_L;
};

__device__ __forceinline__ void chunk_moments(const double* __restrict__ stats, int chunk, double inv_L,
                                              float eps, float& mean, float& rstd) {
  const double s0 = stats[2 * chunk], s1 = stats[2 * chunk + 1];
  const double m = s0 * inv_L;
  double var = s1 * inv_L - m * m;
  var = var < 0.0 ? 0.0 : var;
  mean = (float)m;
  rstd = (float)(1.0 / sqrt(var + (double)eps));
}

// ------------------------------------------------------------------------------------------
template <int VEC>
__global__ void __launch_bounds__(kThreads) gn_stats_kernel(const float* __restrict__ x, double* __restrict__ stats,
                                                           long long L, long long shift, long long n_local) {
  // slab form: x holds the flat elements [shift, shift + n_local) of the sample; a CTA covers the part of its
  // chunk that lies inside (shift = 0, n_local = everything otherwise)
  const int chunk = blockIdx.y;
  const long long e_lo = max(0LL, shift - (long long)chunk * L), e_hi = min(L, shift + n_local - (long long)chunk * L);
  if (e_lo >= e_hi) return;
  const float* xc = x + ((long long)chunk * L - shift);
  float s[2] = {0.f, 0.f};
  // reducing kernels walk several segments per CTA so that few CTAs contend on one fp64 atomic; all kIter loads
  // of a step are issued before the first use
  for (long long base = (long long)blockIdx.x * (kThreads * kIter * VEC); base < L;
       base += (long long)gridDim.x * (kThreads * kIter * VEC)) {
    float v[kIter][VEC];
#pragma unroll
    for (int k = 0; k < kIter; ++k) {
      const long long e = base + ((long long)k * kThreads + threadIdx.x) * VEC;
      const bool in = e >= e_lo && e < e_hi;
      if (VEC == 4) {
        float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
        if (in) t = ld_stream(reinterpret_cast<const float4*>(xc + e));
        v[k][0] = t.x; v[k][VEC > 1 ? 1 : 0] = t.y; v[k][VEC > 2 ? 2 : 0] = t.z; v[k][VEC > 3 ? 3 : 0] = t.w;
      } else {
        v[k][0] = in ? xc[e] : 0.f;
      }
    }
#pragma unroll
    for (int k = 0; k < kIter; ++k)
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        s[0] += v[k][i];
        s[1] += v[k][i] * v[k][i];
      }
  }
  __shared__ double red[64];
  double d[2] = {(double)s[0], (double)s[1]};
  block_sum<2, double>(d, red);
  if (threadIdx.x == 0) {
    atomicAdd(&stats[2 * chunk], d[0]);
    atomicAdd(&stats[2 * chunk + 1], d[1]);
  }
}

// ------------------------------------------------------------------------------------------
template <int VEC, bool RELU>
__global__ void __launch_bounds__(kThreads)
    gn_apply_kernel(const float* __restrict__ x, const double* __restrict__ stats, const float* __restrict__ gamma,
                    const float* __restrict__ beta, float* __restrict__ y, ChunkGeom gm, float eps,
                    long long shift, long long n_local) {
  const int chunk = blockIdx.y;
  const int g = chunk % gm.G;
  const long long e_lo = max(0LL, shift - (long long)chunk * gm.L),
                  e_hi = min(gm.L, shift + n_local - (long long)chunk * gm.L);   // slab form, see gn_stats_kernel
  if (e_lo >= e_hi) return;
  float mean, rstd;
  chunk_moments(stats, chunk, 1.0 / (double)gm.L, eps, mean, rstd);
  const long long off = (long long)chunk * gm.L - shift;
  const long long base = (long long)blockIdx.x * (kThreads * kIter * VEC);
  const int jbase = g * gm.cg;
  const long long goff = (long long)g * gm.L;
  // affine index of element e: (goff + e) % cg.  When cg | kThreads*VEC it is the same for every element a thread
  // touches, so scale = rstd*gamma_j and beta_j are fetched once (no per-element modulo / loads)
  const bool invariant = ((kThreads * VEC) % gm.cg) == 0;
  float sc[4] = {0.f, 0.f, 0.f, 0.f}, sh[4] = {0.f, 0.f, 0.f, 0.f};
  if (invariant) {
    const int c_first = (int)((goff + base + threadIdx.x * VEC) % gm.cg);
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      const int j = (c_first + i) % gm.cg;
      sc[i] = rstd * __ldg(gamma + jbase + j);
      sh[i] = __ldg(beta + jbase + j);
    }
  }
  float in[kIter][4];
#pragma unroll
  for (int k = 0; k < kIter; ++k) {
    const long long e = base + ((long long)k * kThreads + threadIdx.x) * VEC;
    if (e >= e_lo && e < e_hi) {
      if (VEC == 4) {
        const float4 v = ld_stream(reinterpret_cast<const float4*>(x + off + e));
        in[k][0] = v.x; in[k][1] = v.y; in[k][2] = v.z; in[k][3] = v.w;
      } else {
        in[k][0] = x[off + e];
      }
    }
  }
#pragma unroll
  for (int k = 0; k < kIter; ++k) {
    const long long e = base + ((long long)k * kThreads + threadIdx.x) * VEC;
    if (e >= e_lo && e < e_hi) {
      float o[4];
      if (invariant) {
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
          const float t = fmaf(in[k][i] - mean, sc[i], sh[i]);     // (x - mean) first: no cancellation
          o[i] = RELU ? fmaxf(t, 0.f) : t;
        }
      } else {
        const int c0 = (int)((goff + e) % gm.cg);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
          int j = c0 + i;
          j = j >= gm.cg ? j % gm.cg : j;
          const float t = (in[k][i] - mean) * rstd * __ldg(gamma + jbase + j) + __ldg(beta + jbase + j);
          o[i] = RELU ? fmaxf(t, 0.f) : t;
        }
      }
      if (VEC == 4) st_stream(reinterpret_cast<float4*>(y + off + e), make_float4(o[0], o[1], o[2], o[3]));
      else y[off + e] = o[0];
    }
  }
}

// ------------------------------------------------------------------------------------------
// backward pass 1: per chunk  S1 = sum h, S2 = sum h*xhat  (h = dy*[y>0]*gamma_j) -> csum fp64;
//                  per affine index  dgamma_j += sum dy*[y>0]*xhat,  dbeta_j += sum dy*[y>0].
// Fast path needs cg | (kThreads*VEC) so that a thread's affine indices are loop-invariant.
template <int VEC, bool RELU>
__global__ void __launch_bounds__(kThreads)
    gn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ x, const double* __restrict__ stats,
                         const float* __restrict__ gamma, const float* __restrict__ beta,
                         float* __restrict__ dgamma, float* __restrict__ dbeta, double* __restrict__ csum,
                         ChunkGeom gm, float eps) {
  extern __shared__ float sm[];  // [2*cg] + reduction scratch
  float* sg = sm;
  float* sb = sm + gm.cg;
  for (int i = threadIdx.x; i < 2 * gm.cg; i += kThreads) sm[i] = 0.f;
  __syncthreads();
  const int chunk = blockIdx.y;
  const int g = chunk % gm.G;
  float mean, rstd;
  chunk_moments(stats, chunk, 1.0 / (double)gm.L, eps, mean, rstd);
  const long long off = (long long)chunk * gm.L;
  const int jbase = g * gm.cg;
  const long long goff = (long long)g * gm.L;
  const bool invariant = ((kThreads * VEC) % gm.cg) == 0;
  float s1 = 0.f, s2 = 0.f;
  float ag[VEC], ab[VEC];
#pragma unroll
  for (int i = 0; i < VEC; ++i) ag[i] = ab[i] = 0.f;
  // affine index of this thread's first element: loop-invariant when cg | kThreads*VEC
  const int c_first = (int)((goff + (long long)blockIdx.x * (kThreads * kIterR * VEC) + threadIdx.x * VEC) % gm.cg);
  for (long long base = (long long)blockIdx.x * (kThreads * kIterR * VEC); base < gm.L;
       base += (long long)gridDim.x * (kThreads * kIterR * VEC)) {
    // all loads of the step are issued before any use (memory-level parallelism: 2*kIterR 128-bit loads / thread)
    float dv[kIterR][4], xv[kIterR][4];
#pragma unroll
    for (int k = 0; k < kIterR; ++k) {
      const long long e = base + ((long long)k * kThreads + threadIdx.x) * VEC;
#pragma unroll
      for (int i = 0; i < 4; ++i) dv[k][i] = xv[k][i] = 0.f;
      if (e < gm.L) {
        if (VEC == 4) {
          const float4 a = ld_stream(reinterpret_cast<const float4*>(dy + off + e));
          const float4 b = ld_stream(reinterpret_cast<const float4*>(x + off + e));
          dv[k][0] = a.x, dv[k][1] = a.y, dv[k][2] = a.z, dv[k][3] = a.w;
          xv[k][0] = b.x, xv[k][1] = b.y, xv[k][2] = b.z, xv[k][3] = b.w;
        } else {
          dv[k][0] = dy[off + e];
          xv[k][0] = x[off + e];
        }
      }
    }
#pragma unroll
    for (int k = 0; k < kIterR; ++k) {
      const long long e = base + ((long long)k * kThreads + threadIdx.x) * VEC;
      if (e < gm.L) {
        const int c0 = invariant ? c_first : (int)((goff + e) % gm.cg);
#pragma unroll
        for (int i = 0; i < VEC; ++i) {
          int j = c0 + i;
          j = j >= gm.cg ? j % gm.cg : j;
          const float ga = __ldg(gamma + jbase + j);
          const float xh = (xv[k][i] - mean) * rstd;
          float gq = dv[k][i];
          if (RELU) gq = (xh * ga + __ldg(beta + jbase + j)) > 0.f ? gq : 0.f;
          const float h = gq * ga;
          s1 += h;
          s2 += h * xh;
          if (invariant) {
            ag[i] += gq * xh;
            ab[i] += gq;
          } else {
            atomicAdd(&sg[j], gq * xh);
            atomicAdd(&sb[j], gq);
          }
        }
      }
    }
  }
  if (invariant) {
    // lanes whose first elements are congruent mod cg hold the same affine indices: for power-of-two cg <= 128 that
    // is every P = max(1, cg/VEC)-th lane, so a butterfly over the lane offsets >= P leaves the warp totals in
    // lanes [0, P) and only those touch shared memory
    int P = 32;
    if ((gm.cg & (gm.cg - 1)) == 0 && gm.cg <= 32 * VEC) P = gm.cg / VEC > 0 ? gm.cg / VEC : 1;
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      float a = ag[i], b = ab[i];
      for (int o = 16; o >= P; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b += __shfl_xor_sync(0xffffffffu, b, o);
      }
      if ((threadIdx.x & 31) < P) {
        const int j = (c_first + i) % gm.cg;
        atomicAdd(&sg[j], a);
        atomicAdd(&sb[j], b);
      }
    }
  }
  __shared__ double red[64];
  double d[2] = {(double)s1, (double)s2};
  block_sum<2, double>(d, red);  // contains __syncthreads -> smem atomics above are complete
  if (threadIdx.x == 0) {
    atomicAdd(&csum[2 * chunk], d[0]);
    atomicAdd(&csum[2 * chunk + 1], d[1]);
  }
  for (int j = threadIdx.x; j < gm.cg; j += kThreads) {
    atomicAdd(&dgamma[jbase + j], sg[j]);
    atomicAdd(&dbeta[jbase + j], sb[j]);
  }
}

// backward pass 2: dx = rstd * (h - S1/L - xhat * S2/L)
template <int VEC, bool RELU>
__global__ void __launch_bounds__(kThreads)
    gn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x, const double* __restrict__ stats,
                        const float* __restrict__ gamma, const float* __restrict__ beta,
                        const double* __restrict__ csum, float* __restrict__ dx, ChunkGeom gm, float eps) {
  const int chunk = blockIdx.y;
  const int g = chunk % gm.G;
  float mean, rstd;
  chunk_moments(stats, chunk, 1.0 / (double)gm.L, eps, mean, rstd);
  const float m1 = (float)(csum[2 * chunk] / (double)gm.L);
  const float m2 = (float)(csum[2 * chunk + 1] / (double)gm.L);
  const long long off = (long long)chunk * gm.L;
  const long long base = (long long)blockIdx.x * (kThreads * kIter * VEC);
  const int jbase = g * gm.cg;
  const long long goff = (long long)g * gm.L;
  const bool invariant = ((kThreads * VEC) % gm.cg) == 0;       // see gn_apply_kernel
  const int c_first = (int)((goff + base + threadIdx.x * VEC) % gm.cg);
  float gai[4] = {0.f, 0.f, 0.f, 0.f}, bei[4] = {0.f, 0.f, 0.f, 0.f};
  if (invariant) {
#pragma unroll
    for (int i = 0; i < VEC; ++i) {
      gai[i] = __ldg(gamma + jbase + (c_first + i) % gm.cg);
      bei[i] = __ldg(beta + jbase + (c_first + i) % gm.cg);
    }
  }
#pragma unroll
  for (int k = 0; k < kIter; ++k) {
    const long long e = base + ((long long)k * kThreads + threadIdx.x) * VEC;
    if (e < gm.L) {
      const int c0 = invariant ? c_first : (int)((goff + e) % gm.cg);
      float dv[4], xv[4], o[4];
      if (VEC == 4) {
        const float4 a = ld_stream(reinterpret_cast<const float4*>(dy + off + e));
        const float4 b = ld_stream(reinterpret_cast<const float4*>(x + off + e));
        dv[0] = a.x, dv[1] = a.y, dv[2] = a.z, dv[3] = a.w;
        xv[0] = b.x, xv[1] = b.y, xv[2] = b.z, xv[3] = b.w;
      } else {
        dv[0] = dy[off + e];
        xv[0] = x[off + e];
      }
#pragma unroll
      for (int i = 0; i < VEC; ++i) {
        float ga, be;
        if (invariant) {
          ga = gai[i]; be = bei[i];
        } else {
          int j = c0 + i;
          j = j >= gm.cg ? j % gm.cg : j;
          ga = __ldg(gamma + jbase + j);
          be = __ldg(beta + jbase + j);
        }
        const float xh = (xv[i] - mean) * rstd;
        float gq = dv[i];
        if (RELU) gq = (xh * ga + be) > 0.f ? gq : 0.f;
        o[i] = rstd * (gq * ga - m1 - xh * m2);
      }
      if (VEC == 4)
        st_stream(reinterpret_cast<float4*>(dx + off + e), make_float4(o[0], o[1], o[2], o[3]));
      else
        dx[off + e] = o[0];
    }
  }
}

// ================================================================================================ P16 twin forms
// GroupNorm apply / backward-apply that write the 16-bit operand twins the tcgen05 convs consume ([B, D, H, C/8, W, 8],
// common.cuh) — one thread = one 16-byte CELL (8 consecutive channels of a voxel): two 128-bit loads per input tensor,
// one 128-bit store per twin, consecutive lanes = consecutive cells of the fp32 tensor, so the reads are contiguous and
// the stores of a warp fall into C/8 plane rows as 16*32/(C/8)-byte runs.  The position inside the twin is computed
// once per thread and advanced by the loop stride (no division in the streaming loop); grids are capped (grid-stride
// loop) so that the per-CTA bias-gradient atomics stay few.
constexpr int kCell = 8;               // elements per thread and step
constexpr int kIter16 = 4;             // cells per thread per CTA pass

// y = act((x - mean) * rstd * gamma_j + beta_j) -> twins (+ optional fp32 y).  grid (gx, chunks), grid-stride inside
// the chunk.  Requires L % 8 == 0 and cg | 8 or 8 | cg (affine indices of a cell are loop-invariant per thread).
template <bool RELU>
__global__ void __launch_bounds__(kThreads)
    gn_apply16_kernel(const float* __restrict__ x, const double* __restrict__ stats, const float* __restrict__ gamma,
                      const float* __restrict__ beta, float* __restrict__ y, ChunkGeom gm, float eps, Twin16 tw,
                      long long shift, long long n_local, int chunk0) {
  pdl_trigger();
  pdl_wait();
  // depth-slab form (n_local >= 0; batch 1): x / y / the twin hold the flat elements [shift, shift + n_local) of the
  // volume whose chunks gm describes; a CTA covers the part of its chunk that lies inside (the grid starts at the
  // first chunk that intersects: chunk0)
  const int chunk = blockIdx.y + chunk0, g = chunk % gm.G, b = chunk / gm.G;
  long long e_lo = 0, e_hi = gm.L;
  if (n_local >= 0) {
    e_lo = max(0LL, shift - (long long)chunk * gm.L);
    e_hi = min(gm.L, shift + n_local - (long long)chunk * gm.L);
    if (e_lo >= e_hi) return;
  } else {
    shift = 0;
  }
  float mean, rstd;
  chunk_moments(stats, chunk, 1.0 / (double)gm.L, eps, mean, rstd);
  const long long off = (long long)chunk * gm.L - shift;
  const long long goff = (long long)g * gm.L;
  // a pass of the grid covers gridDim.x * kIter16 * kThreads cells; a thread's k-th cell of a pass is kThreads cells on
  const long long pass = (long long)gridDim.x * (kIter16 * kThreads * kCell);
  long long e0 = e_lo + ((long long)blockIdx.x * (kIter16 * kThreads) + threadIdx.x) * kCell;
  // affine constants of this thread's 8 channels (invariant: all strides are multiples of cg)
  float sc[8], sh[8];
  {
    const int c_first = (int)((goff + e0) % gm.cg);
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int j = g * gm.cg + (c_first + i) % gm.cg;
      sc[i] = rstd * __ldg(gamma + j);
      sh[i] = __ldg(beta + j);
    }
  }
  CellPos pos = cell_pos(tw, (unsigned)b, (unsigned long long)(goff + e0 - shift), kThreads,
                         (unsigned long long)(pass / kCell) - (kIter16 - 1) * kThreads);
  for (; e0 < e_hi; e0 += pass) {
    float in[kIter16][8];
#pragma unroll
    for (int k = 0; k < kIter16; ++k) {
      const long long e = e0 + (long long)k * (kThreads * kCell);
      if (e < e_hi) {
        ld8(x + off + e, in[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < kIter16; ++k) {
      const long long e = e0 + (long long)k * (kThreads * kCell);
      if (e < e_hi) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float t = fmaf(in[k][i] - mean, sc[i], sh[i]);
          o[i] = RELU ? fmaxf(t, 0.f) : t;
        }
        if (y != nullptr) st8(y + off + e, o);
        cell_store(tw, pos, o);
      }
      if (k < kIter16 - 1) cell_step(tw, pos, pos.dr1, pos.dw1);
      else cell_step(tw, pos, pos.dr2, pos.dw2);
    }
  }
}

// dx = rstd * (h - S1/L - xhat * S2/L) -> bf16 twin (+ optional fp32 dx) and dbias[c] += sum_vox dx (the bias gradient
// of the conv that produced x)
template <bool RELU>
__global__ void __launch_bounds__(kThreads)
    gn_bwd_apply16_kernel(const float* __restrict__ dy, const float* __restrict__ x, const double* __restrict__ stats,
                          const float* __restrict__ gamma, const float* __restrict__ beta,
                          const double* __restrict__ csum, float* __restrict__ dx, ChunkGeom gm, float eps, Twin16 tw,
                          float* __restrict__ dbias) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sdb[];      // [C]
  if (dbias != nullptr) {
    for (int i = threadIdx.x; i < gm.C; i += kThreads) sdb[i] = 0.f;
    __syncthreads();
  }
  constexpr int KI = 2;               // cells per thread and pass (4 x 128-bit loads each)
  const int chunk = blockIdx.y, g = chunk % gm.G, b = chunk / gm.G;
  float mean, rstd;
  chunk_moments(stats, chunk, 1.0 / (double)gm.L, eps, mean, rstd);
  const float m1 = (float)(csum[2 * chunk] / (double)gm.L);
  const float m2 = (float)(csum[2 * chunk + 1] / (double)gm.L);
  const long long off = (long long)chunk * gm.L;
  const long long goff = (long long)g * gm.L;
  const long long pass = (long long)gridDim.x * (KI * kThreads * kCell);
  long long e0 = ((long long)blockIdx.x * (KI * kThreads) + threadIdx.x) * kCell;
  const long long e_first = e0;
  float ga[8], be[8], db[8];
  const int c_first = (int)((goff + e0) % gm.cg);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int j = g * gm.cg + (c_first + i) % gm.cg;
    ga[i] = __ldg(gamma + j);
    be[i] = __ldg(beta + j);
    db[i] = 0.f;
  }
  CellPos pos = cell_pos(tw, (unsigned)b, (unsigned long long)(goff + e0), kThreads,
                         (unsigned long long)(pass / kCell) - (KI - 1) * kThreads);
  for (; e0 < gm.L; e0 += pass) {
    float dv[KI][8], xv[KI][8];
#pragma unroll
    for (int k = 0; k < KI; ++k) {
      const long long e = e0 + (long long)k * (kThreads * kCell);
      if (e < gm.L) {
        ld8(dy + off + e, dv[k]);
        ld8(x + off + e, xv[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < KI; ++k) {
      const long long e = e0 + (long long)k * (kThreads * kCell);
      if (e < gm.L) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float xh = (xv[k][i] - mean) * rstd;
          float gq = dv[k][i];
          if (RELU) gq = (xh * ga[i] + be[i]) > 0.f ? gq : 0.f;
          o[i] = rstd * (gq * ga[i] - m1 - xh * m2);
          db[i] += o[i];
        }
        if (dx != nullptr) st8(dx + off + e, o);
        cell_store(tw, pos, o);
      }
      if (k < KI - 1) cell_step(tw, pos, pos.dr1, pos.dw1);
      else cell_step(tw, pos, pos.dr2, pos.dw2);
    }
  }
  if (dbias != nullptr) {
    // a thread's channel octet is the same for all its cells (C8 divides every stride): lanes C8 apart in the warp hold
    // the same octet -> butterfly over those lane offsets, then min(C8, 32) lanes touch shared memory
    const int C8 = gm.C >> 3;
    const int c0 = (int)((goff + e_first) % gm.C);
    const int P = C8 < 32 ? C8 : 32;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float a = db[i];
      for (int o2 = 16; o2 >= P; o2 >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o2);
      if ((threadIdx.x & 31) < P) atomicAdd(&sdb[c0 + i], a);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < gm.C; i += kThreads)
      if (sdb[i] != 0.f) atomicAdd(&dbias[i], sdb[i]);
  }
}

// backward pass 1 in the same cell-per-thread form (8 consecutive channels per thread and step, affine constants and
// per-index accumulators in registers — the element-wise form above re-loads gamma / beta per element and is bound by
// its load/store unit, 37-50 % of the HBM peak):  csum[chunk] = (sum h, sum h*xhat), dgamma_j, dbeta_j.
template <bool RELU>
__global__ void __launch_bounds__(kThreads)
    gn_bwd_reduce8_kernel(const float* __restrict__ dy, const float* __restrict__ x, const double* __restrict__ stats,
                          const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ dgamma,
                          float* __restrict__ dbeta, double* __restrict__ csum, ChunkGeom gm, float eps) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sm[];  // [2*cg]
  for (int i = threadIdx.x; i < 2 * gm.cg; i += kThreads) sm[i] = 0.f;
  __syncthreads();
  const int chunk = blockIdx.y, g = chunk % gm.G;
  float mean, rstd;
  chunk_moments(stats, chunk, 1.0 / (double)gm.L, eps, mean, rstd);
  const long long off = (long long)chunk * gm.L;
  const long long goff = (long long)g * gm.L;
  constexpr int KI = 4;               // cells per thread and pass (4 x 128-bit loads each): 256 B in flight per thread
  const long long pass = (long long)gridDim.x * (KI * kThreads * kCell);
  long long e0 = ((long long)blockIdx.x * (KI * kThreads) + threadIdx.x) * kCell;
  const int c_first = (int)((goff + e0) % gm.cg);
  float ga[8], be[8], ag[8], ab[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int j = g * gm.cg + (c_first + i) % gm.cg;
    ga[i] = __ldg(gamma + j);
    be[i] = __ldg(beta + j);
    ag[i] = ab[i] = 0.f;
  }
  float s1 = 0.f, s2 = 0.f;
  for (; e0 < gm.L; e0 += pass) {
    float dv[KI][8], xv[KI][8];
#pragma unroll
    for (int k = 0; k < KI; ++k) {
      const long long e = e0 + (long long)k * (kThreads * kCell);
#pragma unroll
      for (int i = 0; i < 8; ++i) dv[k][i] = 0.f, xv[k][i] = mean;
      if (e < gm.L) {
        ld8(dy + off + e, dv[k]);
        ld8(x + off + e, xv[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < KI; ++k) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float xh = (xv[k][i] - mean) * rstd;
        float gq = dv[k][i];
        if (RELU) gq = (xh * ga[i] + be[i]) > 0.f ? gq : 0.f;
        const float h = gq * ga[i];
        s1 += h;
        s2 += h * xh;
        ag[i] += gq * xh;
        ab[i] += gq;
      }
    }
  }
  // affine index of accumulator i: (c_first + i) % cg.  cg <= 8 (cg | 8): every thread holds the same index pattern ->
  // fold the 8 accumulators onto cg, warp-sum, one lane adds.  cg = 8*m: lanes m apart share their 8 indices -> butterfly
  // over the lane offsets >= m, lanes [0, m) add.
  const int lane = threadIdx.x & 31;
  if (gm.cg <= 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      if (j < gm.cg) {
        float a = 0.f, b2 = 0.f;
#pragma unroll
        for (int i = 0; i < 8; ++i)
          if ((c_first + i) % gm.cg == j) { a += ag[i]; b2 += ab[i]; }
        a = warp_sum(a);
        b2 = warp_sum(b2);
        if (lane == 0) { atomicAdd(&sm[j], a); atomicAdd(&sm[gm.cg + j], b2); }
      }
    }
  } else {
    const int m = gm.cg >> 3;
    const int P = m < 32 ? m : 32;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      float a = ag[i], b2 = ab[i];
      for (int o = 16; o >= P; o >>= 1) {
        a += __shfl_xor_sync(0xffffffffu, a, o);
        b2 += __shfl_xor_sync(0xffffffffu, b2, o);
      }
      if (lane < P) {
        atomicAdd(&sm[(c_first + i) % gm.cg], a);
        atomicAdd(&sm[gm.cg + (c_first + i) % gm.cg], b2);
      }
    }
  }
  __shared__ double red[64];
  double d[2] = {(double)s1, (double)s2};
  block_sum<2, double>(d, red);  // contains __syncthreads -> smem atomics above are complete
  if (threadIdx.x == 0) {
    atomicAdd(&csum[2 * chunk], d[0]);
    atomicAdd(&csum[2 * chunk + 1], d[1]);
  }
  for (int j = threadIdx.x; j < gm.cg; j += kThreads) {
    atomicAdd(&dgamma[g * gm.cg + j], sm[j]);
    atomicAdd(&dbeta[g * gm.cg + j], sm[gm.cg + j]);
  }
}

// CTAs per chunk for the cell kernels: every thread runs >= kIter16 steps, at most ~3 waves of CTAs in total, and the
// grid-stride (gx * kThreads cells) is a multiple of C8 so that a thread keeps its channel octet
static inline dim3 gn_grid16(const ChunkGeom& gm, int nchunks, int waves = 8) {
  // waves: cap of the grid in CTAs per SM.  Kernels that end in per-CTA atomics on a handful of addresses (the fused bias
  // gradient: C addresses shared by ALL CTAs, ~15 ns per queued same-address atomic) take a smaller grid
  const long long cells = gm.L / kCell;
  long long gx = (cells + (long long)kThreads * kIter16 - 1) / ((long long)kThreads * kIter16);
  long long cap = ((long long)waves * sm_count() + nchunks - 1) / nchunks;
  if (cap < 1) cap = 1;
  if (gx > cap) gx = cap;
  if (gx < 1) gx = 1;
  return dim3((unsigned)gx, (unsigned)nchunks, 1);
}

static int gn_geom(const TView& x, int groups, ChunkGeom* gm, int* nchunks) {
  const int C = (int)x.shape[x.ndim - 1];
  // reference group_norm.py:51-59
  B3D_REQUIRE(groups >= 1 && C >= groups, B3D_ERR_SHAPE,
              "Number of groups (%d) cannot be more than the number of channels (%d).", groups, C);
  B3D_REQUIRE(C % groups == 0, B3D_ERR_SHAPE,
              "Number of groups (%d) must be a multiple of the number of channels (%d).", groups, C);
  const long long B = x.shape[0];
  const long long ns = x.numel / B;
  gm->L = ns / groups;
  gm->C = C;
  gm->cg = C / groups;
  gm->G = groups;
  gm->inv_L = 1.0f / (float)gm->L;
  *nchunks = (int)(B * groups);
  B3D_REQUIRE(*nchunks <= 65535, B3D_ERR_SHAPE, "batch*groups too large");
  return B3D_OK;
}

static inline dim3 gn_grid(const ChunkGeom& gm, int nchunks, int vec, bool reducing = false) {
  const long long per = (long long)kThreads * kIter * vec;
  long long gx = (gm.L + per - 1) / per;
  if (reducing) {                      // grid-stride inside the chunk: <= ~4 waves of CTAs in total
    long long cap = (4LL * sm_count() + nchunks - 1) / nchunks;
    if (cap < 1) cap = 1;
    if (gx > cap) gx = cap;
  }
  return dim3((unsigned)gx, (unsigned)nchunks, 1);
}

static int check_stats(const DLTensor* t, int nchunks, const char* name, TView* v) {
  B3D_TRY(view(t, DT_F64, -1, false, name, v));
  B3D_REQUIRE(v->numel == 2LL * nchunks, B3D_ERR_SHAPE, "%s: expected %d fp64 values, got %lld", name,
              2 * nchunks, (long long)v->numel);
  return B3D_OK;
}

static int check_affine(const DLTensor* t, int C, const char* name, TView* v) {
  B3D_TRY(view(t, DT_F32, 1, false, name, v));
  B3D_REQUIRE(v->numel == C, B3D_ERR_SHAPE, "%s: expected %d values, got %lld", name, C, (long long)v->numel);
  return B3D_OK;
}

// gn_geom for x as a whole (total_vox = 0) or as the window [vox_offset, vox_offset + voxels of x) of a batch-1 volume
// of total_vox voxels (depth-slab inference): gm then describes the chunks of the WHOLE volume, which need not line up
// with the window, and *shift is the window's first element in the volume.
static int gn_window(const TView& x, int groups, long long vox_offset, long long total_vox, ChunkGeom* gm,
                     int* nchunks, long long* shift) {
  B3D_TRY(gn_geom(x, groups, gm, nchunks));
  *shift = 0;
  if (total_vox == 0) return B3D_OK;
  B3D_REQUIRE(x.shape[0] == 1, B3D_ERR_SHAPE, "GroupNorm window: batch 1");
  B3D_REQUIRE(vox_offset >= 0 && vox_offset + x.numel / gm->C <= total_vox, B3D_ERR_SHAPE,
              "GroupNorm window: bad offset / total (%lld, %lld voxels)", vox_offset, total_vox);
  gm->L = total_vox * gm->C / groups;
  gm->inv_L = 1.0f / (float)gm->L;
  *shift = vox_offset * gm->C;
  return B3D_OK;
}

// the cell kernels need whole cells per chunk, power-of-two octet counts dividing the thread block (so that a thread
// keeps its channel octet over the grid-stride loop) and affine indices that repeat within a cell stride
static int cell_ok(const ChunkGeom& gm, const TView& x) {
  const int C8 = gm.C / 8;
  B3D_REQUIRE(gm.C % 8 == 0 && gm.L % 8 == 0 && (C8 & (C8 - 1)) == 0 && C8 <= kThreads &&
                  ((kThreads * kCell) % gm.cg == 0) && (gm.cg % 8 == 0 || 8 % gm.cg == 0) &&
                  (x.numel / x.shape[0]) / 8 < (1LL << 32) && ((uintptr_t)x.p & 15) == 0,
              B3D_ERR_UNSUPPORTED, "GroupNorm twin kernels: C = 8 * 2^k channels, 8 | chunk length (C=%d, L=%lld)", gm.C,
              (long long)gm.L);
  return B3D_OK;
}

}  // namespace b3d

using namespace b3d;

// total_vox = 0: x is the whole tensor; otherwise the window [vox_offset, vox_offset + voxels of x) of a batch-1 volume
// of total_vox voxels, and `stats` receives the window's PARTIAL sums per chunk of the whole volume (see gn_window)
extern "C" int b3d_gn_stats(const DLTensor* x_, DLTensor* stats_, int groups, long long vox_offset, long long total_vox,
                            void* stream) {
  TView x, st;
  ChunkGeom gm;
  int nchunks;
  long long shift;
  B3D_TRY(view(x_, DT_F32, -1, false, "x", &x));
  B3D_TRY(gn_window(x, groups, vox_offset, total_vox, &gm, &nchunks, &shift));
  B3D_TRY(check_stats(stats_, nchunks, "stats", &st));
  cudaStream_t s = (cudaStream_t)stream;
  B3D_TRY(cuda_ok(cudaMemsetAsync(st.p, 0, sizeof(double) * 2 * nchunks, s), "memset stats"));
  const bool v4 = (gm.L % 4 == 0) && (shift % 4 == 0) && (((uintptr_t)x.p & 15) == 0);
  if (v4)
    gn_stats_kernel<4><<<gn_grid(gm, nchunks, 4, true), kThreads, 0, s>>>((const float*)x.p, (double*)st.p, gm.L, shift,
                                                                          x.numel);
  else
    gn_stats_kernel<1><<<gn_grid(gm, nchunks, 1, true), kThreads, 0, s>>>((const float*)x.p, (double*)st.p, gm.L, shift,
                                                                          x.numel);
  B3D_LAUNCH_CHECK("gn_stats");
  return B3D_OK;
}

// With the twin y16 (and y16b) given: the cell kernel, y nullable; otherwise the element kernel, y required.  The
// window as in b3d_gn_stats, with `stats` the (all-reduced) statistics of the whole volume.
extern "C" int b3d_gn_apply(const DLTensor* x_, const DLTensor* stats_, const DLTensor* gamma_, const DLTensor* beta_,
                            DLTensor* y_, DLTensor* y16_, DLTensor* y16b_, int groups, float eps, int relu,
                            long long vox_offset, long long total_vox, void* stream) {
  B3D_REQUIRE(y16_ != nullptr || y16b_ == nullptr, B3D_ERR_ARG, "gn_apply: y16b without y16");
  TView x, y, st, ga, be;
  ChunkGeom gm;
  int nchunks;
  long long shift;
  B3D_TRY(view(x_, DT_F32, -1, false, "x", &x));
  if (y_ != nullptr || y16_ == nullptr) {
    B3D_TRY(view(y_, DT_F32, -1, false, "y", &y));
    B3D_REQUIRE(x.numel == y.numel, B3D_ERR_SHAPE, "gn_apply: x/y size mismatch");
  }
  B3D_TRY(gn_window(x, groups, vox_offset, total_vox, &gm, &nchunks, &shift));
  B3D_TRY(check_stats(stats_, nchunks, "stats", &st));
  B3D_TRY(check_affine(gamma_, gm.C, "gamma", &ga));
  B3D_TRY(check_affine(beta_, gm.C, "beta", &be));
  cudaStream_t s = (cudaStream_t)stream;
  if (y16_ == nullptr) {
    const bool v4 = (gm.L % 4 == 0) && (shift % 4 == 0) && ((((uintptr_t)x.p | (uintptr_t)y.p) & 15) == 0);
#define LAUNCH(V, R)                                                                                     \
  gn_apply_kernel<V, R><<<gn_grid(gm, nchunks, V), kThreads, 0, s>>>(                                    \
      (const float*)x.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p, (float*)y.p, gm, eps, shift, \
      x.numel)
    if (v4) {
      if (relu) LAUNCH(4, true); else LAUNCH(4, false);
    } else {
      if (relu) LAUNCH(1, true); else LAUNCH(1, false);
    }
#undef LAUNCH
    B3D_LAUNCH_CHECK("gn_apply");
    return B3D_OK;
  }
  B3D_REQUIRE(((uintptr_t)y.p & 15) == 0, B3D_ERR_SHAPE, "gn_apply: y must be 16-byte aligned");
  B3D_TRY(cell_ok(gm, x));
  B3D_REQUIRE(shift % kCell == 0 && x.numel % kCell == 0, B3D_ERR_LAYOUT, "gn_apply: window not cell-aligned");
  Twin16 tw;
  B3D_TRY(twin_view(y16_, y16b_, x, &tw));
  dim3 grid = gn_grid16(gm, nchunks);
  long long n_local = -1;
  int c0 = 0;
  if (total_vox != 0) {      // only the chunks that intersect the window, each CTA row sized for the part it can hold
    c0 = (int)(shift / gm.L);
    const int nc = (int)((shift + x.numel - 1) / gm.L) - c0 + 1;
    ChunkGeom gl = gm;
    if (x.numel < gl.L) gl.L = (x.numel + kCell - 1) / kCell * kCell;
    grid = gn_grid16(gl, nc);
    n_local = x.numel;
  }
  if (relu)
    launch_pdl(gn_apply16_kernel<true>, grid, kThreads, 0, s, (const float*)x.p, (const double*)st.p, (const float*)ga.p,
               (const float*)be.p, (float*)y.p, gm, eps, tw, shift, n_local, c0);
  else
    launch_pdl(gn_apply16_kernel<false>, grid, kThreads, 0, s, (const float*)x.p, (const double*)st.p, (const float*)ga.p,
               (const float*)be.p, (float*)y.p, gm, eps, tw, shift, n_local, c0);
  B3D_LAUNCH_CHECK("gn_apply16");
  return B3D_OK;
}

extern "C" int b3d_gn_bwd_reduce(const DLTensor* dy_, const DLTensor* x_, const DLTensor* stats_,
                                 const DLTensor* gamma_, const DLTensor* beta_, DLTensor* dgamma_,
                                 DLTensor* dbeta_, DLTensor* csum_, int groups, float eps, int relu, void* stream) {
  TView x, dy, st, ga, be, dga, dbe, cs;
  ChunkGeom gm;
  int nchunks;
  B3D_TRY(view(x_, DT_F32, -1, false, "x", &x));
  B3D_TRY(view(dy_, DT_F32, -1, false, "dy", &dy));
  B3D_REQUIRE(x.numel == dy.numel, B3D_ERR_SHAPE, "gn_bwd_reduce: x/dy size mismatch");
  B3D_TRY(gn_geom(x, groups, &gm, &nchunks));
  B3D_TRY(check_stats(stats_, nchunks, "stats", &st));
  B3D_TRY(check_stats(csum_, nchunks, "csum", &cs));
  B3D_TRY(check_affine(gamma_, gm.C, "gamma", &ga));
  B3D_TRY(check_affine(beta_, gm.C, "beta", &be));
  B3D_TRY(check_affine(dgamma_, gm.C, "dgamma", &dga));
  B3D_TRY(check_affine(dbeta_, gm.C, "dbeta", &dbe));
  cudaStream_t s = (cudaStream_t)stream;
  B3D_TRY(cuda_ok(cudaMemsetAsync(cs.p, 0, sizeof(double) * 2 * nchunks, s), "memset csum"));
  B3D_TRY(cuda_ok(cudaMemsetAsync(dga.p, 0, sizeof(float) * gm.C, s), "memset dgamma"));
  B3D_TRY(cuda_ok(cudaMemsetAsync(dbe.p, 0, sizeof(float) * gm.C, s), "memset dbeta"));
  const bool v4 = (gm.L % 4 == 0) && ((((uintptr_t)x.p | (uintptr_t)dy.p) & 15) == 0);
  const size_t smem = sizeof(float) * 2 * gm.cg;
  // cell-per-thread form: whole cells per chunk, affine indices that repeat with the loop stride (a thread keeps them
  // in registers), and cg a power of two (the lane butterfly)
  const bool cells = v4 && gm.L % 8 == 0 && (kThreads * kCell) % gm.cg == 0 && (gm.cg & (gm.cg - 1)) == 0 &&
                     (gm.cg <= 8 || gm.cg % 8 == 0);
  if (cells) {
    if (relu)
      launch_pdl(gn_bwd_reduce8_kernel<true>, gn_grid16(gm, nchunks), kThreads, smem, s, (const float*)dy.p, (const float*)x.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p,
          (float*)dga.p, (float*)dbe.p, (double*)cs.p, gm, eps);
    else
      launch_pdl(gn_bwd_reduce8_kernel<false>, gn_grid16(gm, nchunks), kThreads, smem, s, (const float*)dy.p, (const float*)x.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p,
          (float*)dga.p, (float*)dbe.p, (double*)cs.p, gm, eps);
    B3D_LAUNCH_CHECK("gn_bwd_reduce8");
    return B3D_OK;
  }
#define LAUNCH(V, R)                                                                                       \
  gn_bwd_reduce_kernel<V, R><<<gn_grid(gm, nchunks, V, true), kThreads, smem, s>>>(                              \
      (const float*)dy.p, (const float*)x.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p, \
      (float*)dga.p, (float*)dbe.p, (double*)cs.p, gm, eps)
  if (v4) {
    if (relu) LAUNCH(4, true); else LAUNCH(4, false);
  } else {
    if (relu) LAUNCH(1, true); else LAUNCH(1, false);
  }
#undef LAUNCH
  B3D_LAUNCH_CHECK("gn_bwd_reduce");
  return B3D_OK;
}

// With the twin dx16 given: the cell kernel, dx nullable, and dbias (nullable, fp32 [C]) = column sums of dx = the bias
// gradient of the conv that produced x; otherwise the element kernel, dx required.
extern "C" int b3d_gn_bwd_apply(const DLTensor* dy_, const DLTensor* x_, const DLTensor* stats_,
                                const DLTensor* gamma_, const DLTensor* beta_, const DLTensor* csum_,
                                DLTensor* dx_, DLTensor* dx16_, DLTensor* dbias_, int groups, float eps, int relu,
                                void* stream) {
  B3D_REQUIRE(dx_ != nullptr || dx16_ != nullptr, B3D_ERR_ARG, "gn_bwd_apply: neither dx nor dx16 given");
  B3D_REQUIRE(dbias_ == nullptr || dx16_ != nullptr, B3D_ERR_ARG, "gn_bwd_apply: dbias without dx16");
  TView x, dy, dx, st, ga, be, cs;
  ChunkGeom gm;
  int nchunks;
  B3D_TRY(view(x_, DT_F32, -1, false, "x", &x));
  B3D_TRY(view(dy_, DT_F32, -1, false, "dy", &dy));
  if (dx_ != nullptr) B3D_TRY(view(dx_, DT_F32, -1, false, "dx", &dx));
  B3D_REQUIRE(x.numel == dy.numel && (dx_ == nullptr || x.numel == dx.numel), B3D_ERR_SHAPE,
              "gn_bwd_apply: size mismatch");
  B3D_TRY(gn_geom(x, groups, &gm, &nchunks));
  B3D_TRY(check_stats(stats_, nchunks, "stats", &st));
  B3D_TRY(check_stats(csum_, nchunks, "csum", &cs));
  B3D_TRY(check_affine(gamma_, gm.C, "gamma", &ga));
  B3D_TRY(check_affine(beta_, gm.C, "beta", &be));
  cudaStream_t s = (cudaStream_t)stream;
  if (dx16_ == nullptr) {
    const bool v4 =
        (gm.L % 4 == 0) && ((((uintptr_t)x.p | (uintptr_t)dy.p | (uintptr_t)dx.p) & 15) == 0);
#define LAUNCH(V, R)                                                                                       \
  gn_bwd_apply_kernel<V, R><<<gn_grid(gm, nchunks, V), kThreads, 0, s>>>(                                  \
      (const float*)dy.p, (const float*)x.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p, \
      (const double*)cs.p, (float*)dx.p, gm, eps)
    if (v4) {
      if (relu) LAUNCH(4, true); else LAUNCH(4, false);
    } else {
      if (relu) LAUNCH(1, true); else LAUNCH(1, false);
    }
#undef LAUNCH
    B3D_LAUNCH_CHECK("gn_bwd_apply");
    return B3D_OK;
  }
  B3D_REQUIRE((((uintptr_t)dy.p | (uintptr_t)dx.p) & 15) == 0, B3D_ERR_SHAPE,
              "gn_bwd_apply: dy / dx must be 16-byte aligned");
  B3D_TRY(cell_ok(gm, x));
  Twin16 tw;
  B3D_TRY(twin_view(dx16_, nullptr, x, &tw));
  float* db = nullptr;
  if (dbias_ != nullptr) {
    TView dbv;
    B3D_TRY(check_affine(dbias_, gm.C, "dbias", &dbv));
    db = (float*)dbv.p;
    B3D_TRY(cuda_ok(cudaMemsetAsync(db, 0, sizeof(float) * gm.C, s), "memset dbias"));
  }
  const size_t smem = db != nullptr ? sizeof(float) * gm.C : 0;
  if (relu)
    launch_pdl(gn_bwd_apply16_kernel<true>, gn_grid16(gm, nchunks, db != nullptr ? 3 : 8), kThreads, smem, s, (const float*)dy.p, (const float*)x.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p,
        (const double*)cs.p, (float*)dx.p, gm, eps, tw, db);
  else
    launch_pdl(gn_bwd_apply16_kernel<false>, gn_grid16(gm, nchunks, db != nullptr ? 3 : 8), kThreads, smem, s, (const float*)dy.p, (const float*)x.p, (const double*)st.p, (const float*)ga.p, (const float*)be.p,
        (const double*)cs.p, (float*)dx.p, gm, eps, tw, db);
  B3D_LAUNCH_CHECK("gn_bwd_apply16");
  return B3D_OK;
}
