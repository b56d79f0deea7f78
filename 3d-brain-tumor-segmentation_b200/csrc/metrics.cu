// b3d — evaluation of one whole-volume segmentation: label map, per-region confusion counts, region surfaces, exact
// squared Euclidean distance transforms of the surfaces and the 95th-percentile Hausdorff distance (include/b3d.h).
//
// Every entry point works on the given stream only, allocates nothing and never synchronises with the host, so the
// four calls of one evaluation can be captured in a CUDA graph.  Accumulators live in caller-owned tensors and are
// cleared by the call that fills them.
#include <math.h>

#include "common.cuh"

using namespace b3d;

namespace {

constexpr int kMaxRegions = 8;
constexpr int kMaxLine = 1024;   // longest line of the distance transform on any axis

// ---- label map ----------------------------------------------------------------------------------------------------
// label = first argmax + 1 where the maximum is > threshold, else 0 (the hard decision of dice_coeff_kernel).
template <int C>
__global__ void __launch_bounds__(256)
    label_map_kernel(const float* __restrict__ p, uint8_t* __restrict__ lab, int H, int W, int h, int w,
                     long long n, float thr) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const long long z = i / ((long long)h * w);
    const int rem = (int)(i - z * h * w), y = rem / w, x = rem - y * w;
    const float* q = p + ((z * H + y) * W + x) * C;
    float mx = __ldg(q);
    int am = 0;
#pragma unroll
    for (int c = 1; c < C; ++c) {
      const float v = __ldg(q + c);
      if (v > mx) { mx = v; am = c; }   // first maximum, like tf.argmax
    }
    lab[i] = mx > thr ? (uint8_t)(am + 1) : (uint8_t)0;
  }
}

// ---- confusion counts + surfaces ----------------------------------------------------------------------------------
// Region bits of a label map at (z, y, x) and whether that voxel is on the region's surface: a voxel of region r with a
// 6-neighbour outside r, voxels outside the volume counting as outside.
__device__ __forceinline__ unsigned surface_bits(const uint8_t* __restrict__ m, const uint8_t* lut, long long i, int z,
                                                 int y, int x, int D, int H, int W, unsigned* bits) {
  const long long HW = (long long)H * W;
  const unsigned b = lut[__ldg(m + i)];
  unsigned inner = b;
  inner &= x > 0 ? lut[__ldg(m + i - 1)] : 0u;
  inner &= x < W - 1 ? lut[__ldg(m + i + 1)] : 0u;
  inner &= y > 0 ? lut[__ldg(m + i - W)] : 0u;
  inner &= y < H - 1 ? lut[__ldg(m + i + W)] : 0u;
  inner &= z > 0 ? lut[__ldg(m + i - HW)] : 0u;
  inner &= z < D - 1 ? lut[__ldg(m + i + HW)] : 0u;
  *bits = b;
  return b & ~inner;
}

__global__ void __launch_bounds__(256)
    region_surface_kernel(const uint8_t* __restrict__ pred, const uint8_t* __restrict__ truth,
                          const uint8_t* __restrict__ lut_g, unsigned long long* __restrict__ counts,
                          uint8_t* __restrict__ surf_p, uint8_t* __restrict__ surf_t, int D, int H, int W, int R) {
  __shared__ uint8_t lut[256];
  __shared__ unsigned long long acc[kMaxRegions * 4];
  const unsigned keep = (1u << R) - 1u;
  for (int i = threadIdx.x; i < 256; i += blockDim.x) lut[i] = (uint8_t)(lut_g[i] & keep);
  for (int i = threadIdx.x; i < R * 4; i += blockDim.x) acc[i] = 0ull;
  __syncthreads();
  unsigned cnt[kMaxRegions * 4];
#pragma unroll
  for (int k = 0; k < kMaxRegions * 4; ++k) cnt[k] = 0u;
  const long long n = (long long)D * H * W;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int z = (int)(i / ((long long)H * W));
    const int rem = (int)(i - (long long)z * H * W), y = rem / W, x = rem - y * W;
    unsigned bp, bt;
    surf_p[i] = (uint8_t)surface_bits(pred, lut, i, z, y, x, D, H, W, &bp);
    surf_t[i] = (uint8_t)surface_bits(truth, lut, i, z, y, x, D, H, W, &bt);
#pragma unroll
    for (int r = 0; r < kMaxRegions; ++r) {
      const unsigned a = (bp >> r) & 1u, b = (bt >> r) & 1u;
      cnt[r * 4 + 0] += a & b;           // TP
      cnt[r * 4 + 1] += a & (b ^ 1u);    // FP
      cnt[r * 4 + 2] += (a ^ 1u) & b;    // FN
      cnt[r * 4 + 3] += (a | b) ^ 1u;    // TN
    }
  }
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int k = 0; k < kMaxRegions * 4; ++k) {
    if (k >= R * 4) break;
    unsigned v = __reduce_add_sync(0xffffffffu, cnt[k]);
    if (lane == 0 && v) atomicAdd(&acc[k], (unsigned long long)v);
  }
  __syncthreads();
  for (int k = threadIdx.x; k < R * 4; k += blockDim.x)
    if (acc[k]) atomicAdd(&counts[k], acc[k]);
}

// ---- separable squared Euclidean distance transform -------------------------------------------------------------
// One thread per line, TL lines per CTA.  The CTA stages its lines in shared memory with coalesced accesses (lines of
// the innermost axis are contiguous rows; lines of the outer axes are neighbours in memory), then every thread builds
// the lower envelope of the parabolas f(v) + s^2 (q - v)^2 of its line's finite sites (Felzenszwalb & Huttenlocher)
// and evaluates it.  Intersections are compared by cross-multiplication in fp64: with unit spacing every operand is an
// integer below 2^24, the products stay below 2^53, and the envelope and its values are exact.
//
// Line L starts at (L / inner) * outer_stride + L % inner and its element q lies q * stride further.
//
// FIRST: the input is the surface bit field (uint8) and f = 0 where bit r is set, +inf elsewhere.
template <bool FIRST>
__global__ void edt_pass_kernel(const uint8_t* __restrict__ surf, float* edt, int n, long long lines, long long inner,
                                long long outer_stride, long long stride, long long nvox, double s2) {
  extern __shared__ __align__(16) unsigned char sm_raw[];
  const int TL = blockDim.x, t = threadIdx.x;
  const int P = n | 1;                                   // odd row pitch: lock-step threads hit distinct banks
  float* buf = reinterpret_cast<float*>(sm_raw);         // [TL][P] the lines
  float* env_f = buf + (size_t)TL * P;                   // [n][TL] f at the envelope's sites
  uint16_t* env_v = reinterpret_cast<uint16_t*>(env_f + (size_t)n * TL);   // [n][TL] the sites
  const int r = blockIdx.y;
  float* field = edt + (long long)r * nvox;
  const long long L0 = (long long)blockIdx.x * TL;
  const int nl = (int)(lines - L0 < TL ? lines - L0 : TL);

  __shared__ long long lbase[32];
  if (t < nl) {
    const long long L = L0 + t;
    lbase[t] = (L / inner) * outer_stride + L % inner;
  }
  __syncthreads();
  // stage: rows of the innermost axis walk along the row, other lines walk across them (consecutive lines are
  // neighbours in memory), so consecutive threads touch consecutive addresses either way
  if (stride == 1) {
    for (int li = 0; li < nl; ++li)
      for (int q = t; q < n; q += TL)
        buf[li * P + q] = FIRST ? ((__ldg(surf + lbase[li] + q) >> r) & 1u ? 0.f : INFINITY) : field[lbase[li] + q];
  } else if (t < nl) {
    for (int q = 0; q < n; ++q)
      buf[t * P + q] = FIRST ? ((__ldg(surf + lbase[t] + q * stride) >> r) & 1u ? 0.f : INFINITY)
                             : field[lbase[t] + q * stride];
  }
  __syncthreads();

  if (t < nl) {
    float* line = buf + t * P;
    const double inv = 1.0 / s2;
    // h(v) = f(v) / s^2 + v^2; the parabolas of sites a < b meet at (h(b) - h(a)) / (2 (b - a))
    int k = -1;
    double hk = 0.0, hk1 = 0.0;   // h of envelope entries k and k - 1
    for (int q = 0; q < n; ++q) {
      const float fq = line[q];
      if (!(fq < INFINITY)) continue;
      const double hq = (double)fq * inv + (double)q * q;
      while (k >= 1) {
        const int v1 = env_v[k * TL + t], v0 = env_v[(k - 1) * TL + t];
        // drop site v1 when q's parabola overtakes it no later than v1 overtakes v0
        if ((hq - hk) * (double)(v1 - v0) <= (hk - hk1) * (double)(q - v1)) {
          --k;
          hk = hk1;
          if (k >= 1) {
            const int v = env_v[(k - 1) * TL + t];
            hk1 = (double)env_f[(k - 1) * TL + t] * inv + (double)v * v;
          }
        } else {
          break;
        }
      }
      ++k;
      env_v[k * TL + t] = (uint16_t)q;
      env_f[k * TL + t] = fq;
      hk1 = hk;
      hk = hq;
    }
    if (k < 0) {
      for (int q = 0; q < n; ++q) line[q] = INFINITY;
    } else {
      int j = 0;
      int vj = env_v[t];
      float fj = env_f[t];
      double hj = (double)fj * inv + (double)vj * vj;
      for (int q = 0; q < n; ++q) {
        while (j < k) {
          const int vn = env_v[(j + 1) * TL + t];
          const float fn = env_f[(j + 1) * TL + t];
          const double hn = (double)fn * inv + (double)vn * vn;
          if (hn - hj < 2.0 * (double)q * (double)(vn - vj)) {   // the next parabola is lower from before q on
            ++j; vj = vn; fj = fn; hj = hn;
          } else {
            break;
          }
        }
        const double d = (double)(q - vj);
        line[q] = (float)((double)fj + s2 * d * d);
      }
    }
  }
  __syncthreads();
  if (stride == 1) {
    for (int li = 0; li < nl; ++li)
      for (int q = t; q < n; q += TL) field[lbase[li] + q] = buf[li * P + q];
  } else if (t < nl) {
    for (int q = 0; q < n; ++q) field[lbase[t] + q * stride] = buf[t * P + q];
  }
}

int edt_lines_per_cta(int n) { return n <= 512 ? 32 : 16; }
size_t edt_smem(int n) {
  const int TL = edt_lines_per_cta(n);
  return (size_t)TL * (n | 1) * sizeof(float) + (size_t)n * TL * (sizeof(float) + sizeof(uint16_t));
}
// The opt-in must cover every supported line length: the most is not at kMaxLine (n = 512 with 32 lines per CTA needs
// 64 bytes more than n = 1024 with 16).
size_t edt_smem_max() {
  size_t m = 0;
  for (int n = 1; n <= kMaxLine; ++n) m = edt_smem(n) > m ? edt_smem(n) : m;
  return m;
}

// ---- HD95: exact order statistics by radix select ------------------------------------------------------------------
// Workspace (uint32): hdr[R][8] | hist[R][256] | list[R][2 * nvox].  hdr: 0 list length, 1 surface voxels of the
// prediction, 2 selected prefix, 3 remaining rank, 4 rank lo, 5 next order statistic is equal to the lo one,
// 6 smallest value above the lo one.
enum { H_N = 0, H_NA, H_PREFIX, H_K, H_LO, H_HI_EQ, H_MIN_GT, kHdr = 8 };

// Squared distances at the surface voxels: prediction surface -> truth EDT, truth surface -> prediction EDT, appended
// to the region's list (fp32 bit patterns, which order like uint32 because they are >= 0).
__global__ void __launch_bounds__(256)
    hd_gather_kernel(const uint32_t* __restrict__ edt_t, const uint8_t* __restrict__ surf_p,
                     const uint32_t* __restrict__ edt_p, const uint8_t* __restrict__ surf_t, uint32_t* ws, int R,
                     long long nvox) {
  const int lane = threadIdx.x & 31;
  uint32_t* list0 = ws + R * (kHdr + 256);
  const long long n_round = (nvox + 31) & ~31LL;   // whole warps stay in the loop for the ballots
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_round;
       i += (long long)gridDim.x * blockDim.x) {
    const bool in = i < nvox;
    const unsigned sp = in ? __ldg(surf_p + i) : 0u, st = in ? __ldg(surf_t + i) : 0u;
    if (__ballot_sync(0xffffffffu, (sp | st) != 0u) == 0u) continue;
    for (int r = 0; r < R; ++r) {
      const bool a = (sp >> r) & 1u, b = (st >> r) & 1u;
      const unsigned ma = __ballot_sync(0xffffffffu, a), mb = __ballot_sync(0xffffffffu, b);
      const int na = __popc(ma), nab = na + __popc(mb);
      if (nab == 0) continue;
      uint32_t base = 0;
      if (lane == 0) {
        base = atomicAdd(&ws[r * kHdr + H_N], (uint32_t)nab);
        if (na) atomicAdd(&ws[r * kHdr + H_NA], (uint32_t)na);
      }
      base = __shfl_sync(0xffffffffu, base, 0);
      const unsigned below = (1u << lane) - 1u;
      uint32_t* list = list0 + (long long)r * 2 * nvox;
      if (a) list[base + __popc(ma & below)] = __ldg(edt_t + (long long)r * nvox + i);
      if (b) list[base + na + __popc(mb & below)] = __ldg(edt_p + (long long)r * nvox + i);
    }
  }
}

// Histogram of digit `pass` (8 bits, most significant first) over the list entries whose higher digits equal the
// prefix selected so far.
__global__ void __launch_bounds__(256) hd_hist_kernel(uint32_t* ws, int R, long long nvox, int pass) {
  __shared__ uint32_t h[256];
  const int r = blockIdx.y;
  h[threadIdx.x] = 0u;
  __syncthreads();
  const uint32_t* hdr = ws + r * kHdr;
  const uint32_t n = hdr[H_N], prefix = hdr[H_PREFIX];
  const uint32_t* list = ws + R * (kHdr + 256) + (long long)r * 2 * nvox;
  const int sh = 24 - 8 * pass;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t x = list[i];
    if (pass == 0 || (x >> (sh + 8)) == prefix) atomicAdd(&h[(x >> sh) & 255u], 1u);
  }
  __syncthreads();
  if (h[threadIdx.x]) atomicAdd(&ws[R * kHdr + r * 256 + threadIdx.x], h[threadIdx.x]);
}

// Picks the bucket that holds the remaining rank, extends the prefix and clears the histogram.  Pass 0 sets the rank
// lo = floor(0.95 (n - 1)); pass 3 leaves the exact lo-th value and whether the next one equals it.
__global__ void __launch_bounds__(256) hd_select_kernel(uint32_t* ws, int R, int pass) {
  const int r = blockIdx.x;
  uint32_t* hdr = ws + r * kHdr;
  uint32_t* hist = ws + R * kHdr + r * 256;
  if (threadIdx.x == 0) {
    const uint32_t n = hdr[H_N];
    if (n > 0) {
      uint32_t k;
      if (pass == 0) {
        k = (uint32_t)floor((double)(n - 1) * 0.95);
        hdr[H_LO] = k;
        hdr[H_PREFIX] = 0u;
      } else {
        k = hdr[H_K];
      }
      uint32_t b = 0, c = 0;
      for (; b < 255u; ++b) {
        if (c + hist[b] > k) break;
        c += hist[b];
      }
      k -= c;
      hdr[H_K] = k;
      hdr[H_PREFIX] = (hdr[H_PREFIX] << 8) | b;
      if (pass == 3) {
        const uint32_t lo = hdr[H_LO];
        const uint32_t count_le = (lo - k) + hist[b];   // entries <= the lo-th value
        hdr[H_HI_EQ] = (lo + 1 >= n || lo + 1 < count_le) ? 1u : 0u;
        hdr[H_MIN_GT] = 0xffffffffu;
      }
    }
  }
  __syncthreads();
  hist[threadIdx.x] = 0u;
}

// Smallest list entry above the lo-th value: the next order statistic when it differs from the lo-th.
__global__ void __launch_bounds__(256) hd_min_above_kernel(uint32_t* ws, int R, long long nvox) {
  const int r = blockIdx.y;
  uint32_t* hdr = ws + r * kHdr;
  const uint32_t n = hdr[H_N], x_lo = hdr[H_PREFIX];
  if (n == 0 || hdr[H_HI_EQ]) return;
  const uint32_t* list = ws + R * (kHdr + 256) + (long long)r * 2 * nvox;
  uint32_t m = 0xffffffffu;
  for (uint32_t i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const uint32_t x = list[i];
    if (x > x_lo && x < m) m = x;
  }
  m = __reduce_min_sync(0xffffffffu, m);
  if ((threadIdx.x & 31) == 0 && m != 0xffffffffu) atomicMin(&hdr[H_MIN_GT], m);
}

__device__ __forceinline__ double ratio(long long a, long long b) { return b == 0 ? 1.0 : (double)a / (double)b; }

// (dice, sensitivity, specificity, hd95) per region.  The percentile interpolates like numpy's "linear" method.
__global__ void hd_finalize_kernel(const long long* __restrict__ counts, const uint32_t* __restrict__ ws,
                                   double* __restrict__ out, int R) {
  const int r = threadIdx.x;
  if (r >= R) return;
  const long long tp = counts[r * 4], fp = counts[r * 4 + 1], fn = counts[r * 4 + 2], tn = counts[r * 4 + 3];
  out[r * 4 + 0] = ratio(2 * tp, 2 * tp + fp + fn);
  out[r * 4 + 1] = ratio(tp, tp + fn);
  out[r * 4 + 2] = ratio(tn, tn + fp);
  const uint32_t* hdr = ws + r * kHdr;
  const uint32_t n = hdr[H_N], na = hdr[H_NA], nb = n - na;
  double hd;
  if (na == 0 && nb == 0) {
    hd = 0.0;
  } else if (na == 0 || nb == 0) {
    hd = INFINITY;
  } else {
    const uint32_t lo_bits = hdr[H_PREFIX], hi_bits = hdr[H_HI_EQ] ? lo_bits : hdr[H_MIN_GT];
    const double a = sqrt((double)__uint_as_float(lo_bits)), b = sqrt((double)__uint_as_float(hi_bits));
    const double h = (double)(n - 1) * 0.95, g = h - floor(h);
    const double diff = b - a;
    hd = g >= 0.5 ? b - diff * (1.0 - g) : a + diff * g;
  }
  out[r * 4 + 3] = hd;
}

int check_map(const DLTensor* t, const char* name, TView* v) {
  B3D_TRY(view(t, DT_U8, 3, false, name, v));
  B3D_REQUIRE(v->numel > 0, B3D_ERR_SHAPE, "%s: empty volume", name);
  return B3D_OK;
}

unsigned grid_for(long long n, int per_sm) {
  const long long cap = (long long)per_sm * sm_count(), g = (n + 255) / 256;
  return (unsigned)(g < 1 ? 1 : (g < cap ? g : cap));
}

}  // namespace

extern "C" int b3d_label_map(const DLTensor* y_pred_, DLTensor* labels_, float threshold, void* stream) {
  TView p, l;
  B3D_TRY(view(y_pred_, DT_F32, 4, false, "y_pred", &p));
  B3D_TRY(view(labels_, DT_U8, 3, false, "labels", &l));
  const int C = (int)p.shape[3];
  B3D_REQUIRE(C >= 1 && C <= 4, B3D_ERR_UNSUPPORTED, "label_map: %d classes unsupported (1..4)", C);
  B3D_REQUIRE(l.shape[0] <= p.shape[0] && l.shape[1] <= p.shape[1] && l.shape[2] <= p.shape[2], B3D_ERR_SHAPE,
              "label_map: labels [%lld,%lld,%lld] larger than y_pred [%lld,%lld,%lld]", (long long)l.shape[0],
              (long long)l.shape[1], (long long)l.shape[2], (long long)p.shape[0], (long long)p.shape[1],
              (long long)p.shape[2]);
  if (l.numel == 0) return B3D_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const int H = (int)p.shape[1], W = (int)p.shape[2], h = (int)l.shape[1], w = (int)l.shape[2];
  const unsigned grid = grid_for(l.numel, 8);
  const float* pp = (const float*)p.p;
  uint8_t* lp = (uint8_t*)l.p;
  switch (C) {
    case 1: label_map_kernel<1><<<grid, 256, 0, s>>>(pp, lp, H, W, h, w, l.numel, threshold); break;
    case 2: label_map_kernel<2><<<grid, 256, 0, s>>>(pp, lp, H, W, h, w, l.numel, threshold); break;
    case 3: label_map_kernel<3><<<grid, 256, 0, s>>>(pp, lp, H, W, h, w, l.numel, threshold); break;
    default: label_map_kernel<4><<<grid, 256, 0, s>>>(pp, lp, H, W, h, w, l.numel, threshold); break;
  }
  B3D_LAUNCH_CHECK("label_map");
  return B3D_OK;
}

extern "C" int b3d_region_surface(const DLTensor* pred_, const DLTensor* true_, const DLTensor* lut_,
                                  DLTensor* counts_, DLTensor* surf_pred_, DLTensor* surf_true_, void* stream) {
  TView pr, tr, lut, cnt, sp, st;
  B3D_TRY(check_map(pred_, "pred", &pr));
  B3D_TRY(check_map(true_, "true", &tr));
  B3D_TRY(check_map(surf_pred_, "surf_pred", &sp));
  B3D_TRY(check_map(surf_true_, "surf_true", &st));
  B3D_TRY(view(lut_, DT_U8, 1, false, "lut", &lut));
  B3D_TRY(view(counts_, DT_I64, 2, false, "counts", &cnt));
  for (int i = 0; i < 3; ++i)
    B3D_REQUIRE(tr.shape[i] == pr.shape[i] && sp.shape[i] == pr.shape[i] && st.shape[i] == pr.shape[i],
                B3D_ERR_SHAPE, "region_surface: pred, true and the surfaces must have one shape");
  B3D_REQUIRE(lut.numel == 256, B3D_ERR_SHAPE, "region_surface: lut must have 256 entries");
  const int R = (int)cnt.shape[0];
  B3D_REQUIRE(R >= 1 && R <= kMaxRegions && cnt.shape[1] == 4, B3D_ERR_SHAPE,
              "region_surface: counts must be int64 [R, 4] with 1 <= R <= %d", kMaxRegions);
  cudaStream_t s = (cudaStream_t)stream;
  B3D_TRY(cuda_ok(cudaMemsetAsync(cnt.p, 0, sizeof(long long) * cnt.numel, s), "memset counts"));
  region_surface_kernel<<<grid_for(pr.numel, 8), 256, 0, s>>>(
      (const uint8_t*)pr.p, (const uint8_t*)tr.p, (const uint8_t*)lut.p, (unsigned long long*)cnt.p, (uint8_t*)sp.p,
      (uint8_t*)st.p, (int)pr.shape[0], (int)pr.shape[1], (int)pr.shape[2], R);
  B3D_LAUNCH_CHECK("region_surface");
  return B3D_OK;
}

extern "C" int b3d_surface_edt(const DLTensor* surf_, DLTensor* edt_, int R, float sd, float sh, float sw,
                               void* stream) {
  TView sf, e;
  B3D_TRY(check_map(surf_, "surf", &sf));
  B3D_TRY(view(edt_, DT_F32, 4, false, "edt", &e));
  B3D_REQUIRE(R >= 1 && R <= kMaxRegions, B3D_ERR_ARG, "surface_edt: R=%d outside 1..%d", R, kMaxRegions);
  B3D_REQUIRE(e.shape[0] == R && e.shape[1] == sf.shape[0] && e.shape[2] == sf.shape[1] && e.shape[3] == sf.shape[2],
              B3D_ERR_SHAPE, "surface_edt: edt must be fp32 [R, D, H, W] of the surface's shape");
  B3D_REQUIRE(sd > 0.f && sh > 0.f && sw > 0.f && sd < INFINITY && sh < INFINITY && sw < INFINITY, B3D_ERR_ARG,
              "surface_edt: spacing must be positive and finite");
  const long long D = sf.shape[0], H = sf.shape[1], W = sf.shape[2], N = D * H * W;
  B3D_REQUIRE(D <= kMaxLine && H <= kMaxLine && W <= kMaxLine, B3D_ERR_UNSUPPORTED,
              "surface_edt: lines up to %d voxels (volume %lld x %lld x %lld)", kMaxLine, D, H, W);
  static bool attr = false;
  if (!attr) {
    B3D_TRY(cuda_ok(cudaFuncSetAttribute(edt_pass_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)edt_smem_max()), "cudaFuncSetAttribute(edt_pass)"));
    B3D_TRY(cuda_ok(cudaFuncSetAttribute(edt_pass_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)edt_smem_max()), "cudaFuncSetAttribute(edt_pass)"));
    attr = true;
  }
  cudaStream_t s = (cudaStream_t)stream;
  const uint8_t* bits = (const uint8_t*)sf.p;
  float* f = (float*)e.p;
  // W (contiguous rows) from the surface bits, then H and D in place
  {
    const int TL = edt_lines_per_cta((int)W);
    const long long lines = D * H;
    edt_pass_kernel<true><<<dim3((unsigned)((lines + TL - 1) / TL), R), TL, edt_smem((int)W), s>>>(
        bits, f, (int)W, lines, 1, W, 1, N, (double)sw * sw);
    B3D_LAUNCH_CHECK("edt_pass_w");
  }
  {
    const int TL = edt_lines_per_cta((int)H);
    const long long lines = D * W;
    edt_pass_kernel<false><<<dim3((unsigned)((lines + TL - 1) / TL), R), TL, edt_smem((int)H), s>>>(
        bits, f, (int)H, lines, W, H * W, W, N, (double)sh * sh);
    B3D_LAUNCH_CHECK("edt_pass_h");
  }
  {
    const int TL = edt_lines_per_cta((int)D);
    const long long lines = H * W;
    edt_pass_kernel<false><<<dim3((unsigned)((lines + TL - 1) / TL), R), TL, edt_smem((int)D), s>>>(
        bits, f, (int)D, lines, H * W, N, H * W, N, (double)sd * sd);
    B3D_LAUNCH_CHECK("edt_pass_d");
  }
  return B3D_OK;
}

extern "C" int b3d_hd95(const DLTensor* edt_true_, const DLTensor* surf_pred_, const DLTensor* edt_pred_,
                        const DLTensor* surf_true_, const DLTensor* counts_, DLTensor* out_, DLTensor* workspace_,
                        void* stream) {
  TView et, sp, ep, st, cnt, out, ws;
  B3D_TRY(view(edt_true_, DT_F32, 4, false, "edt_true", &et));
  B3D_TRY(view(edt_pred_, DT_F32, 4, false, "edt_pred", &ep));
  B3D_TRY(check_map(surf_pred_, "surf_pred", &sp));
  B3D_TRY(check_map(surf_true_, "surf_true", &st));
  B3D_TRY(view(counts_, DT_I64, 2, false, "counts", &cnt));
  B3D_TRY(view(out_, DT_F64, 2, false, "out", &out));
  B3D_TRY(view(workspace_, DT_U8, 1, false, "workspace", &ws));
  const int R = (int)cnt.shape[0];
  B3D_REQUIRE(R >= 1 && R <= kMaxRegions && cnt.shape[1] == 4 && out.shape[0] == R && out.shape[1] == 4,
              B3D_ERR_SHAPE, "hd95: counts int64 [R, 4] and out fp64 [R, 4] with 1 <= R <= %d", kMaxRegions);
  for (int i = 0; i < 3; ++i)
    B3D_REQUIRE(st.shape[i] == sp.shape[i] && et.shape[i + 1] == sp.shape[i] && ep.shape[i + 1] == sp.shape[i],
                B3D_ERR_SHAPE, "hd95: the surfaces and distance transforms must have one shape");
  B3D_REQUIRE(et.shape[0] == R && ep.shape[0] == R, B3D_ERR_SHAPE, "hd95: distance transforms must hold R fields");
  const long long N = sp.numel;
  B3D_REQUIRE(2 * N < (1LL << 32), B3D_ERR_UNSUPPORTED, "hd95: volume of %lld voxels too large", N);
  const long long need = 4LL * R * (kHdr + 256 + 2 * N);
  B3D_REQUIRE(ws.numel >= need, B3D_ERR_SHAPE, "hd95: workspace of %lld bytes, needs %lld", (long long)ws.numel,
              need);
  B3D_REQUIRE(((uintptr_t)ws.p & 15) == 0, B3D_ERR_LAYOUT, "hd95: workspace must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  uint32_t* w = (uint32_t*)ws.p;
  B3D_TRY(cuda_ok(cudaMemsetAsync(w, 0, 4LL * R * (kHdr + 256), s), "memset hd95 workspace"));
  hd_gather_kernel<<<grid_for(N, 8), 256, 0, s>>>((const uint32_t*)et.p, (const uint8_t*)sp.p,
                                                  (const uint32_t*)ep.p, (const uint8_t*)st.p, w, R, N);
  B3D_LAUNCH_CHECK("hd_gather");
  const dim3 g((unsigned)(2 * sm_count() / R + 1), R);
  for (int pass = 0; pass < 4; ++pass) {
    hd_hist_kernel<<<g, 256, 0, s>>>(w, R, N, pass);
    B3D_LAUNCH_CHECK("hd_hist");
    hd_select_kernel<<<R, 256, 0, s>>>(w, R, pass);
    B3D_LAUNCH_CHECK("hd_select");
  }
  hd_min_above_kernel<<<g, 256, 0, s>>>(w, R, N);
  B3D_LAUNCH_CHECK("hd_min_above");
  hd_finalize_kernel<<<1, 32, 0, s>>>((const long long*)cnt.p, w, (double*)out.p, R);
  B3D_LAUNCH_CHECK("hd_finalize");
  return B3D_OK;
}
