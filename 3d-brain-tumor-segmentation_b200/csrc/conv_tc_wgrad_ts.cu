// b3d — weight gradient of the 3x3x3 stride-1 convolution for NARROW outputs (Cout <= 32: the 128^3 and 64^3 levels),
// with the un-shifted operand in TENSOR MEMORY (TS-mode tcgen05.mma) and several MMA-issuing warps.
//
// Why (profiles/r01_umma_rate.txt): a small-N MMA whose A operand comes from shared memory occupies the tensor pipe
// ~39 cycles whatever N is (the 4 KB A tile is fetched at ~105 B/clk), and one warp can issue an MMA only every ~50
// cycles; with A in TMEM and >= 4 issuing warps a N = 16 MMA costs 12 cycles.  In
//     dw[tap][ci][co] = sum_v x[v + tap - 1][ci] * dy[v][co]
// the dy factor is the SAME for all 27 taps of a K step (16 voxels), so the GEMM is turned around:
//     D_tap[co][ci] = sum_v dyT[co][v] * x_tap[v][ci],    M = co (A, TMEM), N = ci (B, shifted halo in smem), K = voxels
//   * dyT: bf16 copy of dy in [voxel block of 8 along w][co][8 voxels] order (cast_bf16_t8_kernel), fetched by TMA as
//     K-major 16-byte cells; one `tcgen05.cp.32x128b.warpx4` per 8-voxel K chunk copies the <= 32 real rows into
//     TMEM (broadcast to the four lane quarters; accumulator rows >= Cout are never read).
//   * x: the same bf16 halo planes as conv_tc_wgrad.cu, now the MN-major B operand; a tap is a start-address offset.
//   * 8 issuing warps: warp w owns the taps t = w (mod 8) of the CTA's tap group and its own 8 TMEM columns for A;
//     cp and mma of one thread execute in issue order, so no cross-warp synchronisation is needed inside a tile.
//   * accumulators D_tap stay in TMEM for the whole kernel (TG * Cin <= 448 columns); the voxel tiles are spread over
//     `nsplit` persistent CTAs per tap group and reduced into dw with fp32 atomics at the end (coalesced over co).
#include "common.cuh"
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace b3d {

constexpr int kTsIssuers = 8;
constexpr int kTsThreads = (2 + kTsIssuers) * 32;      // warp 0: epilogue (TMEM lanes 0..31), warp 1: TMA, 2..9: MMA
constexpr int kTsSmem = 227 * 1024;
constexpr int kTsAccCols = 448;                        // columns 448..511: A tiles (8 per issuing warp)

struct TsParams {
  float* dw;
  int Cin, Cout;
  int TD, TH, TW, HD, HH, HW;      // tile and x-halo extents (voxels)
  int px, px_bytes, py;            // x plane pitch / bytes written by TMA, dyT tile bytes
  int stage_bytes, nstages;
  int ntd, nth, ntw, ntiles, nsplit;
  int D;                           // depth of one sample (dyT folds the batch into its depth dimension)
  int x_p16, x_f16;                // x is a P16 operand (per-plane boxes {8*HW, 1, HH, HD, 1}); its type is fp16
};

__device__ __forceinline__ void tc_mma_ts_bf16(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "r"(a_tmem), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_cp_32x128b(uint32_t dst_tmem, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.32x128b.warpx4 [%0], %1;" ::"r"(dst_tmem), "l"(sdesc) : "memory");
}

template <int TG>
__global__ void __launch_bounds__(kTsThreads, 1)
    conv3_wgrad_ts_kernel(const __grid_constant__ CUtensorMap tmx, const __grid_constant__ CUtensorMap tmy,
                          const TsParams prm) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kTsSmem - 128);
  uint64_t* full = bars;        // [4]  TMA bytes
  uint64_t* empty = bars + 4;   // [4]  one tcgen05.commit per issuing warp
  uint64_t* done = bars + 8;    //      one tcgen05.commit per issuing warp
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int tg = blockIdx.y;                 // tap group
  const int xplanes = prm.Cin / 8;
  constexpr bool allD = TG == 27, allH = TG >= 9, allW = TG >= 3;

  if (threadIdx.x == 0) {
    for (int i = 0; i < prm.nstages; ++i) { mbar_init(smem_u32(&full[i]), 1); mbar_init(smem_u32(&empty[i]), kTsIssuers); }
    mbar_init(smem_u32(done), kTsIssuers);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  int gkd = 0, gkh = 0, gkw = 0;
  if (!allD && allH) gkd = tg;
  if (!allH && allW) { gkd = tg / 3; gkh = tg % 3; }
  if (!allW) { gkd = tg / 9; gkh = (tg / 3) % 3; gkw = tg % 3; }
  const int od = gkd - 1, oh = gkh - 1, ow = gkw - 1;

  if (warp == 1) {
    if (lane == 0) {
      int s = 0, ph = 0;
      const uint32_t bytes = (uint32_t)(xplanes * prm.px_bytes + prm.py);
      for (int tile = blockIdx.x; tile < prm.ntiles; tile += prm.nsplit) {
        int t = tile;
        const int wt = t % prm.ntw; t /= prm.ntw;
        const int ht = t % prm.nth; t /= prm.nth;
        const int dt = t % prm.ntd; t /= prm.ntd;
        const int b = t;
        const int w0 = wt * prm.TW, h0 = ht * prm.TH, d0 = dt * prm.TD;
        mbar_wait(smem_u32(&empty[s]), ph ^ 1);
        const uint32_t fb = smem_u32(&full[s]);
        mbar_expect_tx(fb, bytes);
        const uint32_t xdst = smem_u32(smem + (size_t)s * prm.stage_bytes);
        const uint32_t ydst = xdst + (uint32_t)(xplanes * prm.px);
        for (int p = 0; p < xplanes; ++p) {
          if (prm.x_p16) tma_load_5d(xdst + p * prm.px, &tmx, 4 * (w0 + ow), p, h0 + oh, d0 + od, b, fb);
          else tma_load_5d(xdst + p * prm.px, &tmx, 8 * p, w0 + ow, h0 + oh, d0 + od, b, fb);
        }
        tma_load_5d(ydst, &tmy, 0, 0, w0 / 8, h0, b * prm.D + d0, fb);      // dyT: (8, Cout, W/8, H, B*D)
        if (++s == prm.nstages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp >= 2) {
    // ---- MMA issuers: warp iw owns taps t = iw (mod kTsIssuers) and TMEM columns a_col .. a_col + 7 for its A tile
    const int iw = warp - 2;
    const bool leader = elect_one();
    // D = f32, A = B = bf16, A K-major (TMEM), B MN-major, N = Cin, M = 128
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(prm.Cin >> 3) << 17) |
                           ((128u >> 4) << 24);
    const uint32_t a_col = tmem_base + kTsAccCols + iw * 8;
    int s = 0, ph = 0;
    uint32_t acc = 0;
    const int rowc = prm.HW, planec = prm.HH * prm.HW;
    const uint32_t smem_base = smem_u32(smem);
    const int wblk = prm.TW / 8;
    for (int tile = blockIdx.x; tile < prm.ntiles; tile += prm.nsplit) {
      mbar_wait(smem_u32(&full[s]), ph);
      tc_fence_after();
      const uint32_t xaddr = smem_base + (uint32_t)s * (uint32_t)prm.stage_bytes;
      const uint32_t yaddr = xaddr + (uint32_t)(xplanes * prm.px);
      // B (x halo): K = 16 voxels = 8 along w (16 B apart) x 2 h rows (LBO = halo row pitch), N groups = planes (SBO)
      const uint64_t bdesc0 = make_desc(xaddr, (uint32_t)prm.HW * 16, (uint32_t)prm.px);
      // A (dyT) K chunk = 8 voxels of one (d, h, w block): Cout rows 16 B apart; SBO = 8-row group stride = 128 B
      const uint64_t adesc0 = make_desc(yaddr, 0, 128);
      for (int d = 0; d < prm.TD; ++d)
        for (int h = 0; h < prm.TH; h += 2)
          for (int wb = 0; wb < wblk; ++wb) {
            const uint32_t xcell = (uint32_t)((d * prm.HH + h) * prm.HW + wb * 8);
            const uint32_t ycell = (uint32_t)(((d * prm.TH + h) * wblk + wb) * prm.Cout);      // 16-byte cells
            if (leader) {
              tc_cp_32x128b(a_col, adesc0 + ycell);                                            // voxels of row h
              tc_cp_32x128b(a_col + 4, adesc0 + ycell + (uint32_t)(wblk * prm.Cout));          // voxels of row h+1
#pragma unroll
              for (int t = 0; t < TG; ++t) {
                if ((t % kTsIssuers) != iw) continue;
                const int tkd = allD ? t / 9 : 0;
                const int tkh = allH ? (t / 3) % 3 : 0;
                const int tkw = allW ? t % 3 : 0;
                const uint32_t off = xcell + (uint32_t)(tkd * planec + tkh * rowc + tkw);
                tc_mma_ts_bf16(tmem_base + t * prm.Cin, a_col, bdesc0 + off, idesc, acc);
              }
            }
            acc = 1;
          }
      if (leader) tc_commit(smem_u32(&empty[s]));
      __syncwarp();
      if (++s == prm.nstages) { s = 0; ph ^= 1; }
    }
    if (leader) tc_commit(smem_u32(done));
    __syncwarp();
  } else {
    // ---- warp 0: final reduction of this CTA's partial dw (accumulator row co = TMEM lane co)
    mbar_wait(smem_u32(done), 0);
    tc_fence_after();
    const bool has_tiles = blockIdx.x < prm.ntiles;
    const bool live = has_tiles && lane < prm.Cout;
#pragma unroll 1
    for (int t = 0; t < TG; ++t) {
      const int tap = allD ? t : (TG == 9 ? tg * 9 + t : (TG == 3 ? tg * 3 + t : tg));
      for (int j = 0; j < prm.Cin; j += 16) {
        float v[16];
        tc_ld16(tmem_base + t * prm.Cin + j, v);
        if (live) {
          float* dst = prm.dw + ((size_t)tap * prm.Cin + j) * prm.Cout + lane;       // dw[tap][ci][co], co = lane
#pragma unroll
          for (int i = 0; i < 16; ++i) atomicAdd(dst + (size_t)i * prm.Cout, v[i]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// The kernel handles Cin up to 256, but it only beats conv3_wgrad_tc_kernel where that one wastes most of its M rows:
// measured (tools/conv_bench.py wgrad) 128^3 16->16 544 -> 275 us, 64^3 16->32 112 -> 71 us, but 128^3 32->16
// 589 -> 642 us and 64^3 96->32 185 -> 237 us (three tap groups, each paying the per-K-step TMEM copies).  Re-measured
// in round 2 with P16 operands and 2 / 3 / 4 / 6 issuing warps per CTA instead of 8: 64^3 32->32 128-138 us vs 87 us.
bool tc_wgrad_ts_supported(const WgradGeom& wg) {
  return wg.k == 3 && wg.s == 1 && (wg.nB == 16 || wg.nB == 32) && wg.nA == 16 && wg.Ws % 8 == 0 && wg.bigp % 8 == 0;
}

// x: plain bf16 copy [B, D, H, W, Cin]; dyT: bf16 copy in [B*D][H][W/8][Cout][8] order (launch_cast_bf16_t8)
int launch_conv_wgrad_ts(const WgradGeom& wg, const void* x, const void* dyT, float* dw, cudaStream_t s, int x_p16,
                         int x_f16) {
  B3D_REQUIRE(tc_wgrad_ts_supported(wg), B3D_ERR_UNSUPPORTED, "wgrad (TS): shape not supported");
  B3D_REQUIRE((((uintptr_t)x | (uintptr_t)dyT | (uintptr_t)dw) & 15) == 0, B3D_ERR_LAYOUT, "wgrad (TS): alignment");
  const int Cin = wg.nA, Cout = wg.nB;
  const int TG = 27 * Cin <= kTsAccCols ? 27 : (9 * Cin <= kTsAccCols ? 9 : (3 * Cin <= kTsAccCols ? 3 : 1));
  const int ntg = 27 / TG;
  const bool allD = TG == 27, allH = TG >= 9, allW = TG >= 3;
  const int xpl = Cin / 8;
  static const int cand[][3] = {{1, 4, 8}, {2, 4, 8}, {2, 4, 16}, {2, 8, 16}, {4, 8, 16}, {4, 8, 32}, {4, 16, 32}};
  TsParams p;
  memset(&p, 0, sizeof(p));
  const int budget = kTsSmem - 128;
  bool found = false;
  for (int i = 0; i < (int)(sizeof(cand) / sizeof(cand[0])); ++i) {
    const int TD = cand[i][0], TH = cand[i][1], TW = cand[i][2];
    if (found && (TD > wg.Ds * 2 || TH > wg.Hs * 2 || TW > wg.Ws * 2)) continue;
    if (wg.B > 1 && wg.Ds % TD != 0) continue;      // dyT folds the batch into depth: tiles must not straddle samples
    const int HD = TD + (allD ? 2 : 0), HH = TH + (allH ? 2 : 0), HW = TW + (allW ? 2 : 0);
    const int cells = HD * HH * HW;
    const int px = ((cells * 16 + 127) / 128) * 128, py = TD * TH * TW * Cout * 2;
    // the cp of the last K chunk reads 32 rows (512 B) even when Cout = 16: keep that inside the stage
    const long long stage = (((long long)xpl * px + py + 512 + 127) / 128) * 128;
    for (int ns = 3; ns >= 2; --ns)
      if (ns * stage <= budget) {
        p.TD = TD; p.TH = TH; p.TW = TW; p.HD = HD; p.HH = HH; p.HW = HW;
        p.px = px; p.px_bytes = cells * 16; p.py = py; p.stage_bytes = (int)stage; p.nstages = ns;
        found = true;
        break;
      }
  }
  B3D_REQUIRE(found, B3D_ERR_UNSUPPORTED, "wgrad (TS): no tile fits shared memory (Cin=%d Cout=%d)", Cin, Cout);
  p.dw = dw; p.Cin = Cin; p.Cout = Cout; p.D = wg.Ds; p.x_p16 = x_p16; p.x_f16 = x_f16;
  p.ntd = (wg.Ds + p.TD - 1) / p.TD; p.nth = (wg.Hs + p.TH - 1) / p.TH; p.ntw = (wg.Ws + p.TW - 1) / p.TW;
  p.ntiles = wg.B * p.ntd * p.nth * p.ntw;
  int nsplit = sm_count() / ntg;
  if (nsplit < 1) nsplit = 1;
  if (nsplit > p.ntiles) nsplit = p.ntiles;
  p.nsplit = nsplit;
  EncodeTiledFn enc = tma_encode_fn();
  B3D_REQUIRE(enc != nullptr, B3D_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  CUtensorMap tmx, tmy;
  if (x_p16) {
    B3D_TRY(make_p16_map(&tmx, x, x_f16 ? 0 : 1, wg.B, wg.Db, wg.Hb, wg.Wb, Cin / 8, p.HW, 1, p.HH, p.HD));
  } else {
    const cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)wg.Wb, (cuuint64_t)wg.Hb, (cuuint64_t)wg.Db, (cuuint64_t)wg.B};
    const cuuint64_t st[4] = {(cuuint64_t)wg.bigp * 2, (cuuint64_t)wg.bigp * 2 * wg.Wb,
                              (cuuint64_t)wg.bigp * 2 * wg.Wb * wg.Hb, (cuuint64_t)wg.bigp * 2 * wg.Wb * wg.Hb * wg.Db};
    const cuuint32_t box[5] = {8, (cuuint32_t)p.HW, (cuuint32_t)p.HH, (cuuint32_t)p.HD, 1};
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    const CUresult r = enc(&tmx, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)x, dims, st, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    B3D_REQUIRE(r == CUDA_SUCCESS, B3D_ERR_CUDA, "cuTensorMapEncodeTiled(x) failed (%d)", (int)r);
  }
  {
    const int W8 = wg.Ws / 8;
    const cuuint64_t dims[5] = {8, (cuuint64_t)Cout, (cuuint64_t)W8, (cuuint64_t)wg.Hs, (cuuint64_t)wg.Ds * wg.B};
    const cuuint64_t st[4] = {16, (cuuint64_t)Cout * 16, (cuuint64_t)Cout * 16 * W8, (cuuint64_t)Cout * 16 * W8 * wg.Hs};
    const cuuint32_t box[5] = {8, (cuuint32_t)Cout, (cuuint32_t)(p.TW / 8), (cuuint32_t)p.TH, (cuuint32_t)p.TD};
    const cuuint32_t es[5] = {1, 1, 1, 1, 1};
    const CUresult r = enc(&tmy, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)dyT, dims, st, box, es,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    B3D_REQUIRE(r == CUDA_SUCCESS, B3D_ERR_CUDA, "cuTensorMapEncodeTiled(dyT) failed (%d)", (int)r);
  }
  B3D_TRY(cuda_ok(cudaMemsetAsync(dw, 0, sizeof(float) * 27 * (size_t)Cin * Cout, s), "memset dw"));
  dim3 grid((unsigned)nsplit, (unsigned)ntg, 1);
#define LAUNCH(T)                                                                                              \
  do {                                                                                                         \
    static bool attr = false;                                                                                  \
    if (!attr) {                                                                                               \
      B3D_TRY(cuda_ok(cudaFuncSetAttribute(conv3_wgrad_ts_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                           kTsSmem), "cudaFuncSetAttribute(wgrad_ts)"));                        \
      attr = true;                                                                                             \
    }                                                                                                          \
    conv3_wgrad_ts_kernel<T><<<grid, kTsThreads, kTsSmem, s>>>(tmx, tmy, p);                                   \
  } while (0)
  if (TG == 27) LAUNCH(27);
  else if (TG == 9) LAUNCH(9);
  else if (TG == 3) LAUNCH(3);
  else LAUNCH(1);
#undef LAUNCH
  B3D_LAUNCH_CHECK("conv3_wgrad_ts");
  return B3D_OK;
}

// fp32 [nvox][C] -> bf16 [nvox/8][C][8] (8 consecutive voxels = 8 consecutive w) + optional column sums (bias gradient)
__global__ void __launch_bounds__(256)
    cast_bf16_t8_kernel(const float* __restrict__ src, uint4* __restrict__ dst, long long nblk, int C,
                        float* __restrict__ colsum) {
  extern __shared__ float sm[];
  for (int i = threadIdx.x; i < C; i += blockDim.x) sm[i] = 0.f;
  __syncthreads();
  const int c = threadIdx.x % C, bl = threadIdx.x / C, bpb = blockDim.x / C;
  float acc = 0.f;
  for (long long vb = (long long)blockIdx.x * bpb + bl; vb < nblk && bl < bpb; vb += (long long)gridDim.x * bpb) {
    float v[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = __ldg(src + (vb * 8 + j) * C + c);
    uint4 q;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.x) : "f"(v[1]), "f"(v[0]));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.y) : "f"(v[3]), "f"(v[2]));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.z) : "f"(v[5]), "f"(v[4]));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.w) : "f"(v[7]), "f"(v[6]));
    dst[vb * C + c] = q;
    acc += ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
  }
  if (colsum != nullptr) {
    if (bl < bpb) atomicAdd(&sm[c], acc);
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(&colsum[i], sm[i]);
  }
}

int launch_cast_bf16_t8(const float* src, void* dst, long long nvox, int C, float* colsum, cudaStream_t s) {
  B3D_REQUIRE(nvox % 8 == 0 && C >= 1 && C <= 256, B3D_ERR_UNSUPPORTED, "cast_bf16_t8: voxels %% 8 == 0, C <= 256");
  const long long nblk = nvox / 8;
  const int bpb = 256 / C;
  long long blocks = (nblk + (long long)bpb * 4 - 1) / ((long long)bpb * 4);
  const long long cap = 16LL * sm_count();
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (colsum != nullptr) B3D_TRY(cuda_ok(cudaMemsetAsync(colsum, 0, sizeof(float) * C, s), "memset colsum"));
  cast_bf16_t8_kernel<<<(unsigned)blocks, 256, sizeof(float) * C, s>>>(src, (uint4*)dst, nblk, C, colsum);
  B3D_LAUNCH_CHECK("cast_bf16_t8");
  return B3D_OK;
}

}  // namespace b3d
