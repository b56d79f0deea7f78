// b3d — GroupNormalization with TRUE channel groups on NDHWC storage: the semantics of the reference under
// data_format='channels_first' (layers/group_norm.py:83-124 with axis=1; its GPU default, args.py:121-123), where
// group g of a sample = channels [g*cg, (g+1)*cg) of every voxel — unlike the contiguous-chunk behaviour of the
// channels_last path (norm.cu).  Same HBM-streaming structure: every thread owns a fixed quad of channels (block size
// is a multiple of C/4), 128-bit accesses, register accumulators -> shared memory -> one atomic per CTA and value.
// Also the depth-slab apply (whole-volume statistics, fp32 and / or P16 twin output) of sharded inference, and the
// NCDHW <-> NDHWC re-layout kernels the channels_first API surface needs at the model boundary.
#include "common.cuh"
#include "twin16.cuh"

namespace b3d {

struct CG {
  long long S;       // voxels per sample
  int C, G, cg;      // channels, groups, channels per group
  long long vox_per_cta;
};

__device__ __forceinline__ void group_moments(const double* __restrict__ stats, int bg, double inv_n, float eps,
                                              float& mean, float& rstd) {
  const double m = stats[2 * bg] * inv_n;
  double var = stats[2 * bg + 1] * inv_n - m * m;
  var = var < 0.0 ? 0.0 : var;
  mean = (float)m;
  rstd = (float)(1.0 / sqrt(var + (double)eps));
}

// grid (segments, B); block = vpb * (C/4) threads: thread -> (voxel lane, channel quad)
__global__ void gnc_stats_kernel(const float* __restrict__ x, double* __restrict__ stats, CG g) {
  extern __shared__ float sm[];                  // [G][2]
  const int q = g.C / 4, cq = threadIdx.x % q, vl = threadIdx.x / q, vpb = blockDim.x / q, b = blockIdx.y;
  for (int i = threadIdx.x; i < 2 * g.G; i += blockDim.x) sm[i] = 0.f;
  __syncthreads();
  const long long v0 = (long long)blockIdx.x * g.vox_per_cta, v1 = min(g.S, v0 + g.vox_per_cta);
  float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f};
  const float* xb = x + (long long)b * g.S * g.C + cq * 4;
  for (long long v = v0 + vl; v < v1; v += vpb) {
    const float4 t = ld_stream(reinterpret_cast<const float4*>(xb + v * g.C));
    s0[0] += t.x; s0[1] += t.y; s0[2] += t.z; s0[3] += t.w;
    s1[0] += t.x * t.x; s1[1] += t.y * t.y; s1[2] += t.z * t.z; s1[3] += t.w * t.w;
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gi = (cq * 4 + i) / g.cg;
    atomicAdd(&sm[2 * gi], s0[i]);
    atomicAdd(&sm[2 * gi + 1], s1[i]);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * g.G; i += blockDim.x) atomicAdd(&stats[(long long)b * 2 * g.G + i], (double)sm[i]);
}

template <bool RELU>
__global__ void gnc_apply_kernel(const float* __restrict__ x, const double* __restrict__ stats,
                                 const float* __restrict__ gamma, const float* __restrict__ beta,
                                 float* __restrict__ y, CG g, float eps) {
  const int q = g.C / 4, cq = threadIdx.x % q, vl = threadIdx.x / q, vpb = blockDim.x / q, b = blockIdx.y;
  float a[4], c[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ch = cq * 4 + i;
    float mean, rstd;
    group_moments(stats, b * g.G + ch / g.cg, 1.0 / ((double)g.S * g.cg), eps, mean, rstd);
    a[i] = rstd * gamma[ch];
    c[i] = beta[ch] - mean * a[i];
  }
  const long long v0 = (long long)blockIdx.x * g.vox_per_cta, v1 = min(g.S, v0 + g.vox_per_cta);
  const long long base = (long long)b * g.S * g.C + cq * 4;
  for (long long v = v0 + vl; v < v1; v += vpb) {
    const float4 t = ld_stream(reinterpret_cast<const float4*>(x + base + v * g.C));
    float4 o = make_float4(t.x * a[0] + c[0], t.y * a[1] + c[1], t.z * a[2] + c[2], t.w * a[3] + c[3]);
    if (RELU) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
    st_stream(reinterpret_cast<float4*>(y + base + v * g.C), o);
  }
}

// per channel: dgamma_c += sum gq*xhat, dbeta_c += sum gq  (gq = dy*[y>0]); per (b, group): csum = (sum h, sum h*xhat),
// h = gq*gamma_c, obtained from the CTA's per-channel partial sums
template <bool RELU>
__global__ void gnc_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                      const double* __restrict__ stats, const float* __restrict__ gamma,
                                      const float* __restrict__ beta, float* __restrict__ dgamma,
                                      float* __restrict__ dbeta, double* __restrict__ csum, CG g, float eps) {
  extern __shared__ float sm[];                  // [C][2]
  const int q = g.C / 4, cq = threadIdx.x % q, vl = threadIdx.x / q, vpb = blockDim.x / q, b = blockIdx.y;
  for (int i = threadIdx.x; i < 2 * g.C; i += blockDim.x) sm[i] = 0.f;
  __syncthreads();
  float mean[4], rstd[4], ga[4], be[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ch = cq * 4 + i;
    group_moments(stats, b * g.G + ch / g.cg, 1.0 / ((double)g.S * g.cg), eps, mean[i], rstd[i]);
    ga[i] = gamma[ch];
    be[i] = beta[ch];
  }
  float ag[4] = {0.f, 0.f, 0.f, 0.f}, ab[4] = {0.f, 0.f, 0.f, 0.f};
  const long long v0 = (long long)blockIdx.x * g.vox_per_cta, v1 = min(g.S, v0 + g.vox_per_cta);
  const long long base = (long long)b * g.S * g.C + cq * 4;
  for (long long v = v0 + vl; v < v1; v += vpb) {
    const float4 d4 = ld_stream(reinterpret_cast<const float4*>(dy + base + v * g.C));
    const float4 x4 = ld_stream(reinterpret_cast<const float4*>(x + base + v * g.C));
    const float dv[4] = {d4.x, d4.y, d4.z, d4.w}, xv[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float xh = (xv[i] - mean[i]) * rstd[i];
      float gq = dv[i];
      if (RELU) gq = (xh * ga[i] + be[i]) > 0.f ? gq : 0.f;
      ag[i] += gq * xh;
      ab[i] += gq;
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    atomicAdd(&sm[2 * (cq * 4 + i)], ag[i]);
    atomicAdd(&sm[2 * (cq * 4 + i) + 1], ab[i]);
  }
  __syncthreads();
  for (int ch = threadIdx.x; ch < g.C; ch += blockDim.x) {
    atomicAdd(&dgamma[ch], sm[2 * ch]);
    atomicAdd(&dbeta[ch], sm[2 * ch + 1]);
  }
  for (int gi = threadIdx.x; gi < g.G; gi += blockDim.x) {
    double s1 = 0.0, s2 = 0.0;
    for (int j = 0; j < g.cg; ++j) {
      const int ch = gi * g.cg + j;
      s1 += (double)gamma[ch] * sm[2 * ch + 1];    // sum h       = sum_c gamma_c * dbeta_c
      s2 += (double)gamma[ch] * sm[2 * ch];        // sum h*xhat  = sum_c gamma_c * dgamma_c
    }
    atomicAdd(&csum[2 * (b * g.G + gi)], s1);
    atomicAdd(&csum[2 * (b * g.G + gi) + 1], s2);
  }
}

template <bool RELU>
__global__ void gnc_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                     const double* __restrict__ stats, const float* __restrict__ gamma,
                                     const float* __restrict__ beta, const double* __restrict__ csum,
                                     float* __restrict__ dx, CG g, float eps) {
  const int q = g.C / 4, cq = threadIdx.x % q, vl = threadIdx.x / q, vpb = blockDim.x / q, b = blockIdx.y;
  float mean[4], rstd[4], ga[4], be[4], m1[4], m2[4];
  const double inv_n = 1.0 / ((double)g.S * g.cg);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ch = cq * 4 + i, bg = b * g.G + ch / g.cg;
    group_moments(stats, bg, inv_n, eps, mean[i], rstd[i]);
    ga[i] = gamma[ch];
    be[i] = beta[ch];
    m1[i] = (float)(csum[2 * bg] * inv_n);
    m2[i] = (float)(csum[2 * bg + 1] * inv_n);
  }
  const long long v0 = (long long)blockIdx.x * g.vox_per_cta, v1 = min(g.S, v0 + g.vox_per_cta);
  const long long base = (long long)b * g.S * g.C + cq * 4;
  for (long long v = v0 + vl; v < v1; v += vpb) {
    const float4 d4 = ld_stream(reinterpret_cast<const float4*>(dy + base + v * g.C));
    const float4 x4 = ld_stream(reinterpret_cast<const float4*>(x + base + v * g.C));
    const float dv[4] = {d4.x, d4.y, d4.z, d4.w}, xv[4] = {x4.x, x4.y, x4.z, x4.w};
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float xh = (xv[i] - mean[i]) * rstd[i];
      float gq = dv[i];
      if (RELU) gq = (xh * ga[i] + be[i]) > 0.f ? gq : 0.f;
      o[i] = rstd[i] * (gq * ga[i] - m1[i] - xh * m2[i]);
    }
    st_stream(reinterpret_cast<float4*>(dx + base + v * g.C), make_float4(o[0], o[1], o[2], o[3]));
  }
}

// ---- depth-slab form (slab.py): one rank's slab [1, Dl, H, W, C] normalised with the statistics of the WHOLE volume
// (the all-reduced partial sums of gnc_stats_kernel over every slab; a group holds total_voxels * C/G values) ->
// fp32 y and / or its P16 twin.  One thread = one 16-byte twin cell (8 channels of a voxel), kSlabIter cells per pass
// loaded before any is stored; the block is a multiple of C/8 threads and every stride a multiple of C/8 cells, so a
// thread keeps its channel octet over the grid-stride loop and its 8 scale / shift constants are computed once.
constexpr int kSlabIter = 4;
constexpr int kSlabMaxThreads = 512;    // C <= 4096

template <bool RELU>
__global__ void __launch_bounds__(kSlabMaxThreads)
    gnc_apply_slab_kernel(const float* __restrict__ x, const double* __restrict__ stats,
                          const float* __restrict__ gamma, const float* __restrict__ beta, float* __restrict__ y,
                          Twin16 tw, long long ncells, int cg, double inv_n, float eps) {
  pdl_trigger();
  pdl_wait();
  const unsigned nt = blockDim.x;
  const long long cell0 = (long long)blockIdx.x * (kSlabIter * nt) + threadIdx.x;
  const int c8 = (int)(threadIdx.x % tw.C8);
  float a[8], c[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int ch = c8 * 8 + i;
    float mean, rstd;
    group_moments(stats, ch / cg, inv_n, eps, mean, rstd);
    a[i] = rstd * __ldg(gamma + ch);
    c[i] = __ldg(beta + ch) - mean * a[i];
  }
  const long long pass = (long long)gridDim.x * kSlabIter * nt;      // cells
  CellPos pos = cell_pos(tw, 0u, (unsigned long long)cell0 * 8, nt, (unsigned long long)(pass - (kSlabIter - 1) * nt));
  for (long long k0 = cell0; k0 < ncells; k0 += pass) {
    float in[kSlabIter][8];
#pragma unroll
    for (int k = 0; k < kSlabIter; ++k) {
      const long long cell = k0 + (long long)k * nt;
      if (cell < ncells) ld8(x + cell * 8, in[k]);
    }
#pragma unroll
    for (int k = 0; k < kSlabIter; ++k) {
      const long long cell = k0 + (long long)k * nt;
      if (cell < ncells) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float t = fmaf(in[k][i], a[i], c[i]);
          o[i] = RELU ? fmaxf(t, 0.f) : t;
        }
        if (y != nullptr) st8(y + cell * 8, o);
        if (tw.p != nullptr) cell_store(tw, pos, o);
      }
      if (k < kSlabIter - 1) cell_step(tw, pos, pos.dr1, pos.dw1);
      else cell_step(tw, pos, pos.dr2, pos.dw2);
    }
  }
}

// ---- NCDHW <-> NDHWC: [B, C, S] <-> [B, S, C] through 32x32 shared-memory tiles.
// src [B, R, Cn] -> dst [B, Cn, R]; the voxel dimension (millions) always rides on gridDim.x
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                       long long R, long long Cn, int rows_on_x) {
  __shared__ float tile[32][33];
  const long long b = blockIdx.z;
  const long long r0 = (long long)(rows_on_x ? blockIdx.x : blockIdx.y) * 32;
  const long long c0 = (long long)(rows_on_x ? blockIdx.y : blockIdx.x) * 32;
  const int tx = threadIdx.x % 32, ty = threadIdx.x / 32;
  for (int j = ty; j < 32; j += 8) {
    const long long r = r0 + j, c = c0 + tx;
    tile[j][tx] = (r < R && c < Cn) ? src[(b * R + r) * Cn + c] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const long long c = c0 + j, r = r0 + tx;
    if (r < R && c < Cn) dst[(b * Cn + c) * R + r] = tile[tx][j];
  }
}

static int cgeom(const TView& x, int groups, CG* g, int* threads, dim3* grid) {
  const int C = (int)x.shape[x.ndim - 1];
  const long long B = x.shape[0];
  B3D_REQUIRE(groups >= 1 && C >= groups, B3D_ERR_SHAPE,
              "Number of groups (%d) cannot be more than the number of channels (%d).", groups, C);
  B3D_REQUIRE(C % groups == 0, B3D_ERR_SHAPE,
              "Number of groups (%d) must be a multiple of the number of channels (%d).", groups, C);
  B3D_REQUIRE(C % 4 == 0 && C <= 4096, B3D_ERR_UNSUPPORTED, "channel GroupNorm: channels must be a multiple of 4");
  g->S = x.numel / B / C; g->C = C; g->G = groups; g->cg = C / groups;
  const int q = C / 4;
  *threads = q >= 256 ? q : (256 / q) * q;
  const int vpb = *threads / q;
  long long segs = (g->S + (long long)vpb * 16 - 1) / ((long long)vpb * 16);
  const long long cap = (8LL * sm_count() + B - 1) / B;
  if (segs > cap) segs = cap;
  if (segs < 1) segs = 1;
  g->vox_per_cta = (g->S + segs - 1) / segs;
  *grid = dim3((unsigned)((g->S + g->vox_per_cta - 1) / g->vox_per_cta), (unsigned)B, 1);
  B3D_REQUIRE(B <= 65535, B3D_ERR_SHAPE, "batch too large");
  return B3D_OK;
}

static int vecn(const DLTensor* t, int dtype, long long n, const char* name, TView* v) {
  B3D_TRY(view(t, dtype, -1, false, name, v));
  B3D_REQUIRE(v->numel == n, B3D_ERR_SHAPE, "%s: expected %lld values, got %lld", name, n, (long long)v->numel);
  return B3D_OK;
}

}  // namespace b3d

using namespace b3d;

extern "C" int b3d_gn_channel_stats(const DLTensor* x_, DLTensor* stats_, int groups, void* stream) {
  TView x, st;
  CG g; int threads; dim3 grid;
  B3D_TRY(view(x_, DT_F32, -1, false, "x", &x));
  B3D_TRY(cgeom(x, groups, &g, &threads, &grid));
  B3D_TRY(vecn(stats_, DT_F64, 2LL * x.shape[0] * groups, "stats", &st));
  cudaStream_t s = (cudaStream_t)stream;
  B3D_TRY(cuda_ok(cudaMemsetAsync(st.p, 0, sizeof(double) * st.numel, s), "memset stats"));
  gnc_stats_kernel<<<grid, threads, sizeof(float) * 2 * groups, s>>>((const float*)x.p, (double*)st.p, g);
  B3D_LAUNCH_CHECK("gn_channel_stats");
  return B3D_OK;
}

extern "C" int b3d_gn_channel_apply(const DLTensor* x_, const DLTensor* stats_, const DLTensor* gamma_,
                                    const DLTensor* beta_, DLTensor* y_, int groups, float eps, int relu,
                                    void* stream) {
  TView x, y, st, ga, be;
  CG g; int threads; dim3 grid;
  B3D_TRY(view(x_, DT_F32, -1, false, "x", &x));
  B3D_TRY(view(y_, DT_F32, -1, false, "y", &y));
  B3D_REQUIRE(x.numel == y.numel, B3D_ERR_SHAPE, "gn_channel_apply: x/y size mismatch");
  B3D_TRY(cgeom(x, groups, &g, &threads, &grid));
  B3D_TRY(vecn(stats_, DT_F64, 2LL * x.shape[0] * groups, "stats", &st));
  B3D_TRY(vecn(gamma_, DT_F32, g.C, "gamma", &ga));
  B3D_TRY(vecn(beta_, DT_F32, g.C, "beta", &be));
  cudaStream_t s = (cudaStream_t)stream;
  if (relu)
    gnc_apply_kernel<true><<<grid, threads, 0, s>>>((const float*)x.p, (const double*)st.p, (const float*)ga.p,
                                                    (const float*)be.p, (float*)y.p, g, eps);
  else
    gnc_apply_kernel<false><<<grid, threads, 0, s>>>((const float*)x.p, (const double*)st.p, (const float*)ga.p,
                                                     (const float*)be.p, (float*)y.p, g, eps);
  B3D_LAUNCH_CHECK("gn_channel_apply");
  return B3D_OK;
}

extern "C" int b3d_gn_channel_bwd(const DLTensor* dy_, const DLTensor* x_, const DLTensor* stats_,
                                  const DLTensor* gamma_, const DLTensor* beta_, DLTensor* dgamma_, DLTensor* dbeta_,
                                  DLTensor* csum_, DLTensor* dx_, int groups, float eps, int relu, void* stream) {
  TView x, dy, dx, st, ga, be, dga, dbe, cs;
  CG g; int threads; dim3 grid;
  B3D_TRY(view(x_, DT_F32, -1, false, "x", &x));
  B3D_TRY(view(dy_, DT_F32, -1, false, "dy", &dy));
  B3D_TRY(view(dx_, DT_F32, -1, false, "dx", &dx));
  B3D_REQUIRE(x.numel == dy.numel && x.numel == dx.numel, B3D_ERR_SHAPE, "gn_channel_bwd: size mismatch");
  B3D_TRY(cgeom(x, groups, &g, &threads, &grid));
  const long long nst = 2LL * x.shape[0] * groups;
  B3D_TRY(vecn(stats_, DT_F64, nst, "stats", &st));
  B3D_TRY(vecn(csum_, DT_F64, nst, "csum", &cs));
  B3D_TRY(vecn(gamma_, DT_F32, g.C, "gamma", &ga));
  B3D_TRY(vecn(beta_, DT_F32, g.C, "beta", &be));
  B3D_TRY(vecn(dgamma_, DT_F32, g.C, "dgamma", &dga));
  B3D_TRY(vecn(dbeta_, DT_F32, g.C, "dbeta", &dbe));
  cudaStream_t s = (cudaStream_t)stream;
  B3D_TRY(cuda_ok(cudaMemsetAsync(cs.p, 0, sizeof(double) * nst, s), "memset csum"));
  B3D_TRY(cuda_ok(cudaMemsetAsync(dga.p, 0, sizeof(float) * g.C, s), "memset dgamma"));
  B3D_TRY(cuda_ok(cudaMemsetAsync(dbe.p, 0, sizeof(float) * g.C, s), "memset dbeta"));
  const size_t smem = sizeof(float) * 2 * g.C;
#define B3D_GNC(R)                                                                                              \
  do {                                                                                                          \
    gnc_bwd_reduce_kernel<R><<<grid, threads, smem, s>>>((const float*)dy.p, (const float*)x.p, (const double*)st.p, \
                                                         (const float*)ga.p, (const float*)be.p, (float*)dga.p, \
                                                         (float*)dbe.p, (double*)cs.p, g, eps);                 \
    gnc_bwd_apply_kernel<R><<<grid, threads, 0, s>>>((const float*)dy.p, (const float*)x.p, (const double*)st.p, \
                                                     (const float*)ga.p, (const float*)be.p, (const double*)cs.p, \
                                                     (float*)dx.p, g, eps);                                     \
  } while (0)
  if (relu) B3D_GNC(true); else B3D_GNC(false);
#undef B3D_GNC
  B3D_LAUNCH_CHECK("gn_channel_bwd");
  return B3D_OK;
}

// One depth slab of sharded inference (slab.py): x / y / y16 = this rank's slab [1, Dl, H, W, C] (y16: its P16 twin
// [1, Dl, H, C/8, W, 8]); stats = the all-reduced (sum x, sum x^2) of every channel group over the whole volume of
// total_voxels voxels (total_voxels = the slab's own voxel count: the un-sharded apply).  y and y16 are each optional,
// not both.
extern "C" int b3d_gn_channel_apply_slab(const DLTensor* x_, const DLTensor* stats_, const DLTensor* gamma_,
                                         const DLTensor* beta_, DLTensor* y_, DLTensor* y16_, int groups, float eps,
                                         int relu, long long total_voxels, void* stream) {
  TView x, y, st, ga, be;
  B3D_TRY(view(x_, DT_F32, 5, false, "x", &x));
  B3D_REQUIRE(x.shape[0] == 1, B3D_ERR_SHAPE, "gn_channel_apply (slab): batch 1");
  B3D_REQUIRE(y_ != nullptr || y16_ != nullptr, B3D_ERR_ARG, "gn_channel_apply (slab): neither y nor y16 given");
  const int C = (int)x.shape[4];
  B3D_REQUIRE(groups >= 1 && C >= groups, B3D_ERR_SHAPE,
              "Number of groups (%d) cannot be more than the number of channels (%d).", groups, C);
  B3D_REQUIRE(C % groups == 0, B3D_ERR_SHAPE,
              "Number of groups (%d) must be a multiple of the number of channels (%d).", groups, C);
  B3D_REQUIRE(C % 8 == 0 && C / 8 <= kSlabMaxThreads && ((uintptr_t)x.p & 15) == 0, B3D_ERR_UNSUPPORTED,
              "gn_channel_apply (slab): channels must be a multiple of 8, at most %d (C=%d)", 8 * kSlabMaxThreads, C);
  const long long S = x.numel / C, ncells = x.numel / 8;
  B3D_REQUIRE(S > 0 && total_voxels >= S, B3D_ERR_ARG,
              "gn_channel_apply (slab): total_voxels (%lld) below the slab's %lld voxels", total_voxels, S);
  B3D_REQUIRE(ncells < (1LL << 32), B3D_ERR_UNSUPPORTED, "gn_channel_apply (slab): slab too large");
  y.p = nullptr;
  if (y_ != nullptr) {
    B3D_TRY(view(y_, DT_F32, -1, false, "y", &y));
    B3D_REQUIRE(x.numel == y.numel && ((uintptr_t)y.p & 15) == 0, B3D_ERR_SHAPE,
                "gn_channel_apply (slab): x/y size mismatch");
  }
  B3D_TRY(vecn(stats_, DT_F64, 2LL * groups, "stats", &st));
  B3D_TRY(vecn(gamma_, DT_F32, C, "gamma", &ga));
  B3D_TRY(vecn(beta_, DT_F32, C, "beta", &be));
  // the cell position is advanced for y-only calls too, so its geometry is that of x
  Twin16 tw;
  tw.p = nullptr; tw.p2 = nullptr; tw.bf16 = 0;
  tw.W = (unsigned)x.shape[3]; tw.C8 = (unsigned)(C / 8); tw.rows = (unsigned)(x.shape[1] * x.shape[2]);
  if (y16_ != nullptr) B3D_TRY(twin_view(y16_, nullptr, x, &tw));
  const int q = C / 8;
  const int threads = q >= 256 ? q : (256 / q) * q;
  long long blocks = (ncells + (long long)threads * kSlabIter - 1) / ((long long)threads * kSlabIter);
  const long long cap = 8LL * sm_count();
  if (blocks > cap) blocks = cap;
  const double inv_n = 1.0 / ((double)total_voxels * (C / groups));
  cudaStream_t s = (cudaStream_t)stream;
  if (relu)
    launch_pdl(gnc_apply_slab_kernel<true>, dim3((unsigned)blocks), threads, 0, s, (const float*)x.p,
               (const double*)st.p, (const float*)ga.p, (const float*)be.p, (float*)y.p, tw, ncells, C / groups, inv_n,
               eps);
  else
    launch_pdl(gnc_apply_slab_kernel<false>, dim3((unsigned)blocks), threads, 0, s, (const float*)x.p,
               (const double*)st.p, (const float*)ga.p, (const float*)be.p, (float*)y.p, tw, ncells, C / groups, inv_n,
               eps);
  B3D_LAUNCH_CHECK("gn_channel_apply (slab)");
  return B3D_OK;
}

// to_channels_last = 1: src [B, C, D, H, W] -> dst [B, D, H, W, C];  0: the inverse
extern "C" int b3d_relayout(const DLTensor* src_, DLTensor* dst_, int to_channels_last, void* stream) {
  TView a, b;
  B3D_TRY(view(src_, DT_F32, 5, false, "src", &a));
  B3D_TRY(view(dst_, DT_F32, 5, false, "dst", &b));
  B3D_REQUIRE(a.numel == b.numel && a.shape[0] == b.shape[0], B3D_ERR_SHAPE, "relayout: size mismatch");
  const long long B = a.shape[0];
  const long long C = to_channels_last ? a.shape[1] : a.shape[4];
  B3D_REQUIRE((to_channels_last ? b.shape[4] : b.shape[1]) == C, B3D_ERR_SHAPE, "relayout: channel mismatch");
  const long long S = a.numel / B / C;
  B3D_REQUIRE((C + 31) / 32 <= 65535 && B <= 65535, B3D_ERR_SHAPE, "relayout: too many channels / samples");
  cudaStream_t s = (cudaStream_t)stream;
  const dim3 grid((unsigned)((S + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
  if (to_channels_last)      // src [B, R = C, Cn = S] -> dst [B, S, C]: columns (voxels) on x
    transpose_kernel<<<grid, 256, 0, s>>>((const float*)a.p, (float*)b.p, C, S, 0);
  else                       // src [B, R = S, Cn = C] -> dst [B, C, S]: rows (voxels) on x
    transpose_kernel<<<grid, 256, 0, s>>>((const float*)a.p, (float*)b.p, S, C, 1);
  B3D_LAUNCH_CHECK("relayout");
  return B3D_OK;
}
