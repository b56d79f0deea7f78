// b3d — weight gradient of the 3x3x3 stride-1 SAME convolution on the tcgen05 tensor cores:
//     dw[tap][ci][co] = sum_voxels x[v + tap - 1][ci] * dy[v][co]          (train.py:151, tape.gradient)
// as 27 shifted GEMMs  D_tap[ci][co] += X_tap^T . dY  with the VOXELS as the contraction dimension:
//   * A = x halo tile, B = dy tile, both bf16 (fp32 accumulate) in a 16-byte-cell plane layout
//     plane[c/8][voxel][8 ch], which for a reduction over voxels is the canonical *MN-major*
//     SWIZZLE_NONE UMMA layout (verified on hardware by tools/umma_probe_bf16.cu; kind::tf32 does not
//     accept MN-major SWIZZLE_NONE operands — tools/umma_probe.cu — hence bf16 here):
//     8 consecutive-w voxels = the 8 K-rows of a core matrix (16 B apart), the second K group = the
//     next h row (LBO = row pitch), channel groups of 8 = MN groups one plane apart (SBO = plane
//     bytes).  One MMA contracts 16 voxels for M = 128 input channels x N = Cout, and the tap shift is
//     again only a start-address offset into the resident halo.
//   * the bf16 copies of x and dy are produced by cast_bf16_kernel below (which also emits the bias
//     gradient = column sums of dy), so the tiles can be fetched by TMA.
//   * accumulators D_tap live in TMEM for the whole kernel (TG taps x Cout columns <= 512); taps are
//     split into groups (27 / 9 / 3 / 1 taps) and input channels into tiles of 128 across CTAs; the
//     voxel tiles of one (channel tile, tap group) are spread over `nsplit` persistent CTAs and the
//     partial results are reduced into dw with fp32 atomics at the end (dw pre-zeroed).
//   * the same kernel runs the 1x1x1 weight gradient (KS = 1: one tap, no halo) and the stride-2 family (KS = 2):
//     Conv3D k3 s2 / Conv3DTranspose are 2x2x2 stride-1 convs of the space-to-depth "big" tensor (conv_s2.cu), whose
//     bf16 copy is written directly in [B, D/2, H/2, W/2, 8*C] order by cast_bf16_s2d_kernel; the epilogue scatters
//     the (coarse tap, parity) blocks back to the 27 taps of dw.  Wide `small` tensors are cut into N tiles.
//   * when fewer than 128 input channels remain, the missing MN groups address shared memory past the
//     real planes (still inside this CTA's allocation, enforced by the host planner); the
//     corresponding accumulator rows are never read.
#include <limits.h>

#include "common.cuh"
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace b3d {

__device__ __forceinline__ void tc_mma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}

struct WgParams {
  float* dw;
  int Cin, Cout;                   // rows (virtual big channels) and columns (small channels) of one tap of dw
  int NT, nnt;                     // N tile (columns per CTA) and number of N tiles
  int pad;                         // halo before (1 for k=3, 0 for k in {1,2})
  int s2_nA;                       // > 0: stride-2 family, Cin = 8*s2_nA rows ordered (parity, channel)
  int px_bytes;                    // bytes the TMA writes per x plane (px is the 128-byte padded pitch)
  int M;                           // MMA M: 128, or 64 when <= 64 rows exist (half the A-operand shared-memory reads)
  int rows_real;                   // rows of dw actually written (stacked narrow operands are zero-padded to 8)
  int tr_cn;                       // > 0: rows are (tap, c) of a stacked narrow dy with tr_cn channels and the columns are
                                   //      the layer's input channels: write dw[tap][column][c] (see cast_stack_bf16)
  int TD, TH, TW, HD, HH, HW;      // tile and x-halo extents (voxels)
  int px, py;                      // plane bytes of x halo / dy tile
  int stage_bytes, nstages, xplanes_max;
  int ntd, nth, ntw, ntiles;
  int nsplit;
  // P16 operands (common.cuh): every plane is fetched by its own TMA box {8*HW, 1, HH, HD, 1} from the tensor map of
  // the source that holds it (virtual concat of up to 4 big tensors: cend8 = cumulative channel octets)
  int p16, nsrc;
  int cend8[4];
};

struct alignas(64) WgMaps {
  CUtensorMap x[4];
  CUtensorMap y;
  CUtensorMap y2;      // kd-in-M kernel only: gradient of the block's pointwise conv output (same x, second dw)
};

constexpr int kWgSmem = 227 * 1024;

template <int KS, int TG>
__global__ void __launch_bounds__(256, 1)
    conv3_wgrad_tc_kernel(const __grid_constant__ WgMaps maps, const WgParams prm) {
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t smem[];
  // barriers live at the very end of the allocation (the garbage MN groups never reach them: host planner)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgSmem - 128);
  uint64_t* full = bars;        // [4]
  uint64_t* empty = bars + 4;   // [4]
  uint64_t* done = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int TAPS = KS * KS * KS;
  constexpr bool allD = TG == TAPS, allH = TG >= KS * KS, allW = TG >= KS;   // dims a tap group spans
  const int tg = blockIdx.y;                 // tap group
  const int cbase = (blockIdx.z / prm.nnt) * prm.M;   // input-channel tile
  const int nb0 = (blockIdx.z % prm.nnt) * prm.NT;  // output-channel tile
  const int crem = min(prm.M, prm.Cin - cbase);
  const int xplanes = crem / 8, yplanes = prm.NT / 8;

  if (threadIdx.x == 0) {
    for (int i = 0; i < prm.nstages; ++i) { mbar_init(smem_u32(&full[i]), 1); mbar_init(smem_u32(&empty[i]), 1); }
    mbar_init(smem_u32(done), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // first tap of this group and the halo origin shift it implies
  int gkd = 0, gkh = 0, gkw = 0;
  if (!allD && allH) gkd = tg;
  if (!allH && allW) { gkd = tg / KS; gkh = tg % KS; }
  if (!allW) { gkd = tg / (KS * KS); gkh = (tg / KS) % KS; gkw = tg % KS; }
  const int od = gkd - prm.pad, oh = gkh - prm.pad, ow = gkw - prm.pad;

  if (warp == 0) {
    if (lane == 0) {
      int s = 0, ph = 0;
      const uint32_t bytes = (uint32_t)(xplanes * prm.px_bytes + yplanes * prm.py);
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
        const uint32_t ydst = xdst + (uint32_t)(prm.xplanes_max * prm.px);
        if (prm.p16) {
          for (int p = 0; p < xplanes; ++p) {
            const int gp = (cbase >> 3) + p;
            int si = 0;
            while (si + 1 < prm.nsrc && gp >= prm.cend8[si]) ++si;
            tma_load_5d(xdst + p * prm.px, &maps.x[si], 4 * (w0 + ow), gp - (si > 0 ? prm.cend8[si - 1] : 0), h0 + oh,
                        d0 + od, b, fb);
          }
          for (int q = 0; q < yplanes; ++q)
            tma_load_5d(ydst + q * prm.py, &maps.y, 4 * w0, (nb0 >> 3) + q, h0, d0, b, fb);
        } else {
          for (int p = 0; p < xplanes; ++p)
            tma_load_5d(xdst + p * prm.px, &maps.x[0], cbase + 8 * p, w0 + ow, h0 + oh, d0 + od, b, fb);
          for (int q = 0; q < yplanes; ++q) tma_load_5d(ydst + q * prm.py, &maps.y, nb0 + 8 * q, w0, h0, d0, b, fb);
        }
        if (++s == prm.nstages) { s = 0; ph ^= 1; }
      }
    }
  } else if (warp == 1) {
    // whole warp runs the warp-uniform control flow (descriptors stay in uniform registers); one elected
    // lane issues the MMAs and commits
    const bool leader = elect_one();
    // D=f32, A=B=bf16, both MN-major, N=Cout, M=128
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                           ((uint32_t)(prm.NT >> 3) << 17) | (((uint32_t)prm.M >> 4) << 24);
    int s = 0, ph = 0;
    uint32_t acc = 0;
    const int rowc = prm.HW, planec = prm.HH * prm.HW;
    const uint32_t smem_base = smem_u32(smem);
    for (int tile = blockIdx.x; tile < prm.ntiles; tile += prm.nsplit) {
      mbar_wait(smem_u32(&full[s]), ph);
      tc_fence_after();
      const uint32_t xaddr = smem_base + (uint32_t)s * (uint32_t)prm.stage_bytes;
      // K = 16 voxels per MMA: 8 along w (16 B apart) x 2 h rows (LBO = row pitch of each operand)
      const uint64_t adesc0 = make_desc(xaddr, (uint32_t)prm.HW * 16, (uint32_t)prm.px);
      const uint64_t bdesc0 =
          make_desc(xaddr + (uint32_t)(prm.xplanes_max * prm.px), (uint32_t)prm.TW * 16, (uint32_t)prm.py);
      for (int d = 0; d < prm.TD; ++d)
        for (int h = 0; h < prm.TH; h += 2)
          for (int w8 = 0; w8 < prm.TW; w8 += 8) {
            const uint32_t ycell = (uint32_t)((d * prm.TH + h) * prm.TW + w8);
            const uint32_t xcell = (uint32_t)((d * prm.HH + h) * prm.HW + w8);
            const uint64_t bdesc = bdesc0 + ycell;
            if (leader) {
#pragma unroll
              for (int t = 0; t < TG; ++t) {
                const int tkd = allD ? t / (KS * KS) : 0;
                const int tkh = allH ? (t / KS) % KS : 0;
                const int tkw = allW ? t % KS : 0;
                const uint32_t off = xcell + (uint32_t)(tkd * planec + tkh * rowc + tkw);
                tc_mma_bf16(tmem_base + t * prm.NT, adesc0 + off, bdesc, idesc, acc);
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
  } else if (warp >= 4) {
    // final reduction of this CTA's partial dw into global memory
    // accumulator row r lives in TMEM lane r (M = 128) or lane 32*(r/16) + r%16 (M = 64; tools/umma_probe_m64.cu)
    const int q = warp - 4;
    mbar_wait(smem_u32(done), 0);
    tc_fence_after();
    const bool has_tiles = blockIdx.x < prm.ntiles;
    // A warp's 32 rows x NT columns go through shared memory (the stage buffers are free once `done` fired) so that
    // consecutive lanes add consecutive 16-byte pieces of a dw row (REDG.128): with a row per lane every scalar atomic
    // instruction touched 32 sectors, and the split-K CTAs queued on them for tens of microseconds per launch.
    const int pitch = prm.NT + 4, c4n = prm.NT / 4;
    float* stg = reinterpret_cast<float*>(smem) + q * 32 * pitch;
    const bool vec = prm.tr_cn == 0 && (prm.Cout & 3) == 0;
#pragma unroll 1
    for (int tt = 0; tt < TG; ++tt) {
      const int t = (tt + (int)blockIdx.x) % TG;          // CTAs start at different taps: fewer same-address queues
      const int tap0 = allD ? t : (TG == KS * KS ? tg * TG + t : (TG == KS ? tg * KS + t : tg));
      for (int j = 0; j < prm.NT; j += 16) {
        float v[16];
        tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + t * prm.NT + j, v);
#pragma unroll
        for (int i = 0; i < 16; i += 4)
          *reinterpret_cast<float4*>(stg + lane * pitch + j + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
      __syncwarp();
      // rows of the block: lane-row rl -> input channel (or (parity, channel) / (tap, narrow channel)) row ci
      const int nel = vec ? 32 * c4n : 32 * prm.NT;
      for (int e = lane; has_tiles && e < nel; e += 32) {
        const int rl = vec ? e / c4n : e / prm.NT, c = vec ? (e - rl * c4n) * 4 : e - rl * prm.NT;
        const int ci = prm.M == 128 ? cbase + q * 32 + rl : (rl < 16 ? cbase + q * 16 + rl : prm.Cin);
        if (ci >= prm.rows_real) continue;
        // stride-2 family: row ci = (parity, channel); coarse tap d and parity p give the fine tap 2d + p (<= 2)
        int row = ci, rows = prm.Cin, tap = tap0;
        if (prm.s2_nA > 0) {
          const int par = ci / prm.s2_nA;
          row = ci - par * prm.s2_nA; rows = prm.s2_nA;
          const int td = 2 * (tap0 >> 2) + (par >> 2), th = 2 * ((tap0 >> 1) & 1) + ((par >> 1) & 1),
                    tw = 2 * (tap0 & 1) + (par & 1);
          if (td > 2 || th > 2 || tw > 2) continue;
          tap = (td * 3 + th) * 3 + tw;
        }
        const float* src = stg + rl * pitch + c;
        if (vec) {
          atomicAdd(reinterpret_cast<float4*>(prm.dw + ((size_t)tap * rows + row) * prm.Cout + nb0 + c),
                    *reinterpret_cast<const float4*>(src));
        } else if (prm.tr_cn > 0) {
          const int tr = row / prm.tr_cn, cc = row - tr * prm.tr_cn;     // row = (tap, narrow channel)
          atomicAdd(prm.dw + ((size_t)tr * prm.Cout + nb0 + c) * prm.tr_cn + cc, *src);
        } else {
          atomicAdd(prm.dw + ((size_t)tap * rows + row) * prm.Cout + nb0 + c, *src);
        }
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// N tile (columns of dw per CTA): all taps of a group must fit the 512 TMEM columns
static int wgrad_ntile(int k, int nB) {
  const int cap = k == 2 ? 64 : 256;     // k=2: the 8 coarse taps stay resident (8 * 64 = 512 columns)
  if (nB <= cap) return nB;
  for (int nt = cap; nt >= 16; nt >>= 1)
    if (nB % nt == 0) return nt;
  return 0;
}

bool tc_wgrad_supported(const WgradGeom& wg) {
  const bool kind = (wg.s == 1 && (wg.k == 3 || wg.k == 1)) || (wg.s == 2 && wg.k == 3);
  return kind && wg.nA % 8 == 0 && wg.nA >= 8 && wg.nB % 16 == 0 && wg.nB >= 16 &&
         wgrad_ntile(wg.s == 2 ? 2 : wg.k, wg.nB) > 0 && wg.bigp % 8 == 0 && wg.smallp % 8 == 0;
}

static int make_map(CUtensorMap* tm, const void* base, int C, long long pitch, int W, int H, int D, int B,
                    int bw, int bh, int bd) {
  EncodeTiledFn enc = tma_encode_fn();
  B3D_REQUIRE(enc != nullptr, B3D_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  const cuuint64_t dims[5] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  const cuuint64_t strides[4] = {(cuuint64_t)pitch * 2, (cuuint64_t)pitch * 2 * W, (cuuint64_t)pitch * 2 * W * H,
                                 (cuuint64_t)pitch * 2 * W * H * D};
  const cuuint32_t box[5] = {8, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bd, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, (void*)base, dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B3D_REQUIRE(r == CUDA_SUCCESS, B3D_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d)", (int)r);
  return B3D_OK;
}

// x: bf16 copy of the big tensor — for stride 2 already in space-to-depth order [B, Ds, Hs, Ws, 8*nA]
// rows_real / tr_cn: see WgParams (0 / 0 for ordinary layers); dw_elems: size of dw to clear
int launch_conv_wgrad_tc(const WgradGeom& wg, const void* x, const void* dy, float* dw, cudaStream_t s,
                         int rows_real, int tr_cn, long long dw_elems, const WgP16* p16) {
  B3D_REQUIRE(tc_wgrad_supported(wg), B3D_ERR_UNSUPPORTED, "wgrad: shape not on the tcgen05 path");
  B3D_REQUIRE((((uintptr_t)x | (uintptr_t)dy | (uintptr_t)dw) & 15) == 0, B3D_ERR_LAYOUT, "wgrad: alignment");
  const bool s2 = wg.s == 2;
  B3D_REQUIRE(p16 == nullptr || (rows_real == 0 && tr_cn == 0), B3D_ERR_UNSUPPORTED, "wgrad (P16): plain layers only");
  const int KS = s2 ? 2 : wg.k, TAPS = KS * KS * KS;
  const int Cin = s2 ? 8 * wg.nA : wg.nA, Cout = wg.nB;
  const int NT = wgrad_ntile(KS, Cout), nnt = Cout / NT;
  int TG;
  if (KS == 3) TG = 27 * NT <= 512 ? 27 : (9 * NT <= 512 ? 9 : (3 * NT <= 512 ? 3 : 1));
  else TG = TAPS;
  const int ntg = TAPS / TG;
  const bool allD = TG == TAPS, allH = TG >= KS * KS, allW = TG >= KS;
  const int M = Cin <= 64 ? 64 : 128;
  const int nmt = (Cin + M - 1) / M;
  const int xpl = (Cin < M ? Cin : M) / 8;
  // tile planner: largest tile whose stages fit, with 16 MN groups (M=128 bf16) readable from every stage start
  static const int cand[][3] = {{1, 4, 8},  {2, 4, 8},  {2, 4, 16}, {2, 8, 16},
                                {4, 8, 16}, {4, 8, 32}, {4, 16, 32}};   // TH even: a K step spans 2 h rows
  WgParams p;
  memset(&p, 0, sizeof(p));
  const int budget = kWgSmem - 128;
  bool found = false;
  for (int i = 0; i < (int)(sizeof(cand) / sizeof(cand[0])); ++i) {
    const int TD = cand[i][0], TH = cand[i][1], TW = cand[i][2];
    if (found && (TD > wg.Ds * 2 || TH > wg.Hs * 2 || TW > wg.Ws * 2)) continue;   // do not over-tile tiny volumes
    const int HD = TD + (allD ? KS - 1 : 0), HH = TH + (allH ? KS - 1 : 0), HW = TW + (allW ? KS - 1 : 0);
    const int cells = HD * HH * HW;
    const int px = ((cells * 16 + 127) / 128) * 128, py = TD * TH * TW * 16;
    const long long stage = (((long long)xpl * px + (long long)(NT / 8) * py + 127) / 128) * 128;
    for (int ns = 3; ns >= 2; --ns) {
      const long long last = (long long)(ns - 1) * stage;
      if (ns * stage <= budget && last + (long long)(M / 8) * px <= budget) {
        p.TD = TD; p.TH = TH; p.TW = TW; p.HD = HD; p.HH = HH; p.HW = HW;
        p.px = px; p.px_bytes = cells * 16; p.py = py; p.stage_bytes = (int)stage; p.nstages = ns;
        found = true;
        break;
      }
    }
  }
  B3D_REQUIRE(found, B3D_ERR_UNSUPPORTED, "wgrad: no tile fits shared memory (Cin=%d Cout=%d)", Cin, Cout);
  p.dw = dw; p.Cin = Cin; p.Cout = Cout; p.xplanes_max = xpl;
  p.NT = NT; p.nnt = nnt; p.pad = KS == 3 ? 1 : 0; p.s2_nA = s2 ? wg.nA : 0;
  p.M = M; p.rows_real = rows_real > 0 ? rows_real : Cin; p.tr_cn = tr_cn;
  p.ntd = (wg.Ds + p.TD - 1) / p.TD; p.nth = (wg.Hs + p.TH - 1) / p.TH; p.ntw = (wg.Ws + p.TW - 1) / p.TW;
  p.ntiles = wg.B * p.ntd * p.nth * p.ntw;
  int nsplit = sm_count() / (ntg * nmt * nnt);
  if (nsplit < 1) nsplit = 1;
  if (nsplit > p.ntiles) nsplit = p.ntiles;
  p.nsplit = nsplit;
  WgMaps maps;
  memset(&maps, 0, sizeof(maps));
  if (p16 != nullptr) {
    // big: the sources concatenate to Cin channels (stride 2: ONE coarse space-to-depth tensor with 8*nA channels)
    // kind::f16 takes ONE operand type for A and B (mixing f16 with bf16 is an illegal instruction on sm_100a — tried):
    // the weight gradient reads bf16 twins of both tensors
    B3D_REQUIRE(p16->big_bf16 && p16->small_bf16, B3D_ERR_DTYPE, "wgrad (P16): both operands must be bf16 twins");
    p.p16 = 1; p.nsrc = p16->n;
    int cum = 0;
    for (int i = 0; i < p16->n; ++i) {
      cum += p16->C[i] / 8;
      p.cend8[i] = cum;
      B3D_TRY(make_p16_map(&maps.x[i], p16->big[i], p16->big_bf16, wg.B, s2 ? wg.Ds : wg.Db, s2 ? wg.Hs : wg.Hb,
                           s2 ? wg.Ws : wg.Wb, p16->C[i] / 8, p.HW, 1, p.HH, p.HD));
    }
    B3D_REQUIRE(cum * 8 == Cin, B3D_ERR_SHAPE, "wgrad (P16): sources hold %d channels, expected %d", cum * 8, Cin);
    B3D_TRY(make_p16_map(&maps.y, p16->small, p16->small_bf16, wg.B, wg.Ds, wg.Hs, wg.Ws, Cout / 8, p.TW, 1, p.TH, p.TD));
  } else {
    if (s2) B3D_TRY(make_map(&maps.x[0], x, Cin, Cin, wg.Ws, wg.Hs, wg.Ds, wg.B, p.HW, p.HH, p.HD));
    else    B3D_TRY(make_map(&maps.x[0], x, Cin, wg.bigp, wg.Wb, wg.Hb, wg.Db, wg.B, p.HW, p.HH, p.HD));
    B3D_TRY(make_map(&maps.y, dy, Cout, wg.smallp, wg.Ws, wg.Hs, wg.Ds, wg.B, p.TW, p.TH, p.TD));
  }
  const size_t dw_n = dw_elems > 0 ? (size_t)dw_elems : (size_t)wg.k * wg.k * wg.k * wg.nA * Cout;
  B3D_TRY(cuda_ok(cudaMemsetAsync(dw, 0, sizeof(float) * dw_n, s), "memset dw"));
  dim3 grid((unsigned)nsplit, (unsigned)ntg, (unsigned)(nmt * nnt));
#define LAUNCH(K, T)                                                                                           \
  do {                                                                                                         \
    static bool attr = false;                                                                                  \
    if (!attr) {                                                                                               \
      B3D_TRY(cuda_ok(cudaFuncSetAttribute(conv3_wgrad_tc_kernel<K, T>,                                         \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem),             \
                      "cudaFuncSetAttribute(wgrad_tc)"));                                                      \
      attr = true;                                                                                             \
    }                                                                                                          \
    conv3_wgrad_tc_kernel<K, T><<<grid, 256, kWgSmem, s>>>(maps, p);                                       \
  } while (0)
  if (KS == 1) LAUNCH(1, 1);
  else if (KS == 2) LAUNCH(2, 8);
  else if (TG == 27) LAUNCH(3, 27);
  else if (TG == 9) LAUNCH(3, 9);
  else if (TG == 3) LAUNCH(3, 3);
  else LAUNCH(3, 1);
#undef LAUNCH
  B3D_LAUNCH_CHECK("conv3_wgrad_tc");
  return B3D_OK;
}


// ================================================================================ kd folded into M, kw folded into N
// For Cin = 32 / 64 the kernel above computes M = 64 / 128 rows per MMA of which Cin are real, 27 MMAs per K step.  Here
// the three depth taps share the M dimension and the three width taps the N dimension of ONE MMA:
//   * the x tile (32 or 16 channels, halo in d and h only) is laid out [d][plane][h][w] — ONE TMA box of a tensor map
//     whose dimensions are ordered (w, h, plane, d) when a single source covers the tile's planes, else one box per
//     depth slice and source piece — so the M groups (kd, plane) of the A operand lie at ONE stride (a plane slice):
//     96 of 128 rows (Cin = 32) or 48 of 64 (Cin = 16) are real;
//   * the dy tile is loaded three times, shifted by 1 - kw voxels along w (TMA zero fill at the volume edge), so the N
//     groups (kw, plane) of the B operand lie at one stride as well and
//         D_kh[(kd, ci)][(kw, co)] += sum_u x[u + (kd-1, kh-1, 0)][ci] * dy[u - (0, 0, kw-1)][co]
//     is the weight gradient with the voxel sum re-indexed (u = v + (0, 0, kw-1));
//   * no operand is read at a w offset: every 128-byte core matrix the tensor core fetches from shared memory is
//     aligned (the form with kw as an MMA loop measured ~63 cycles per M = 128, N = 16 MMA, twice its operand bytes).
// 3 MMAs (N = 3 Cout) per K step instead of 27, one per kh tap, each issued by its own warp into its own accumulator
// block (a warp issues a tcgen05.mma only every ~50 cycles); all accumulators (9 Cout <= 288 columns, + Cout for the
// pointwise layer) in one CTA; 32-channel tiles (blockIdx.y) and voxel ranges (blockIdx.x) are spread over the CTAs.
// Warps: 0 TMA producer, 1..3 MMA issuers (2 also owns the TMEM allocation), 4..7 final reduction.
struct KdfParams {
  float* dw;
  float* dw2;                      // != nullptr: also dw of the pointwise conv reading the same x, [Cin][Cout]: one more
                                   // MMA per K step (A = the centre rows of the x tile, B = a tile of its dy)
  int Cin, Cout;
  int TD, TH, TW, HD, HH, HW;
  int pslice;                      // pitch of one (plane, depth slice) of the halo: HH * HW * 16 bytes padded to 128
  int py;                          // bytes of one dy plane of the tile
  int xbytes, stage_bytes, nstages;
  int ntd, nth, ntw, ntiles, nsplit;
  int nsrc, cend8[4];
  int g, xbd;                      // an x box holds g planes x xbd depth slices (xbd = HD when one source covers the
                                   // tile's planes: the whole halo is ONE box; else one box per (depth slice, g planes))
  int P;                           // channel planes (octets) of the tile: 4 (Cin = 32, M = 128) or 2 (Cin = 16, M = 64)
};

__global__ void __launch_bounds__(256, 1)
    conv3_wgrad_kdf_kernel(const __grid_constant__ WgMaps maps, const KdfParams prm) {
  pdl_trigger();
  extern __shared__ __align__(1024) uint8_t smem[];
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kWgSmem - 128);
  uint64_t* full = bars;        // [4]
  uint64_t* empty = bars + 4;   // [4]
  uint64_t* done = bars + 8;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 9);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int P = prm.P;
  const int cbase = blockIdx.y * 8 * P;       // channel tile
  const int yplanes = prm.Cout / 8;

  if (threadIdx.x == 0) {
    // one MMA-issuing warp per kh tap (a warp can issue a tcgen05.mma only every ~50 cycles: profiles/r01_umma_rate.txt)
    for (int i = 0; i < prm.nstages; ++i) { mbar_init(smem_u32(&full[i]), 1); mbar_init(smem_u32(&empty[i]), 3); }
    mbar_init(smem_u32(done), 3);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 2) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // producer warp: lane 0 waits for the slot and arms the barrier, then the lanes issue the tile's boxes in parallel
    int s = 0, ph = 0;
    // boxes of a tile (tensor maps with permuted dimensions: a box is a whole [d][plane][h][w] / [plane][d][h][w] block):
    // x: (HD / xbd) x (P / g); dy: one per copy, all planes; dres: one
    const int pg = P / prm.g, nxb = (prm.HD / prm.xbd) * pg, nyb = 3;
    const int nbox = nxb + nyb + (prm.dw2 != nullptr ? 1 : 0);
    const uint32_t bytes = (uint32_t)(prm.HD * P * prm.HH * prm.HW * 16 + (nbox - nxb) * yplanes * prm.py);
    for (int tile = blockIdx.x; tile < prm.ntiles; tile += prm.nsplit) {
      int t = tile;
      const int wt = t % prm.ntw; t /= prm.ntw;
      const int ht = t % prm.nth; t /= prm.nth;
      const int dt = t % prm.ntd; t /= prm.ntd;
      const int b = t;
      const int w0 = wt * prm.TW, h0 = ht * prm.TH, d0 = dt * prm.TD;
      const uint32_t fb = smem_u32(&full[s]);
      if (lane == 0) {
        mbar_wait(smem_u32(&empty[s]), ph ^ 1);
        mbar_expect_tx(fb, bytes);
      }
      __syncwarp();
      const uint32_t xdst = smem_u32(smem + (size_t)s * prm.stage_bytes);
      const uint32_t ydst = xdst + (uint32_t)prm.xbytes;
      for (int j = lane; j < nbox; j += 32) {
        if (j < nxb) {
          const int d = j / pg, p = (j - d * pg) * prm.g;
          const int gp = (cbase >> 3) + p;
          int si = 0;
          while (si + 1 < prm.nsrc && gp >= prm.cend8[si]) ++si;
          const int lp = gp - (si > 0 ? prm.cend8[si - 1] : 0);
          tma_load_5d(xdst + (uint32_t)((d * P + p) * prm.pslice), &maps.x[si], 4 * w0, h0 - 1, lp, d0 - 1 + d, b, fb);
        } else {
          // dy three times, shifted by 1 - kw voxels along w (zero fill outside the volume): copy kw at in-tile voxel u
          // holds dy[u - (kw - 1)], the partner of x[u + (kd - 1, kh - 1, 0)]
          const int jj = j - nxb;
          if (jj >= nyb) tma_load_5d(ydst + 3 * yplanes * prm.py, &maps.y2, 4 * w0, h0, d0, 0, b, fb);
          else tma_load_5d(ydst + jj * yplanes * prm.py, &maps.y, 4 * (w0 + 1 - jj), h0, d0, 0, b, fb);
        }
      }
      __syncwarp();
      if (++s == prm.nstages) { s = 0; ph ^= 1; }
    }
  } else if (warp >= 1 && warp <= 3) {
    // warps 1..3: the MMAs of kh tap (warp - 1), each into its own accumulator block
    const int t = warp - 1;
    const bool leader = elect_one();
    // D = f32, A = B = bf16, both MN-major, N = 3 Cout (columns (kw, co)), M = 128 / 64 (rows (kd, ci): 96 / 48 real)
    const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                           ((uint32_t)((3 * prm.Cout) >> 3) << 17) | (((uint32_t)(32 * P) >> 4) << 24);
    const uint32_t idesc2 = (1u << 4) | (1u << 7) | (1u << 10) | (1u << 15) | (1u << 16) |
                            ((uint32_t)(prm.Cout >> 3) << 17) | (((uint32_t)(32 * P) >> 4) << 24);
    int s = 0, ph = 0;
    uint32_t acc = 0;
    const uint32_t smem_base = smem_u32(smem);
    const int slicec = prm.pslice / 16;          // cells between consecutive (plane, depth slice) blocks
    for (int tile = blockIdx.x; tile < prm.ntiles; tile += prm.nsplit) {
      mbar_wait(smem_u32(&full[s]), ph);
      tc_fence_after();
      const uint32_t xaddr = smem_base + (uint32_t)s * (uint32_t)prm.stage_bytes;
      // A: K = 8 voxels along w x 2 h rows (LBO = halo row), M groups (kd, plane) one plane slice apart (SBO);
      // B: the same K cells of the three dy copies, N groups (kw, plane) one dy plane apart
      const uint64_t adesc0 = make_desc(xaddr, (uint32_t)prm.HW * 16, (uint32_t)prm.pslice);
      const uint64_t bdesc0 = make_desc(xaddr + (uint32_t)prm.xbytes, (uint32_t)prm.TW * 16, (uint32_t)prm.py);
      const uint64_t bdesc2 = make_desc(xaddr + (uint32_t)(prm.xbytes + 3 * yplanes * prm.py), (uint32_t)prm.TW * 16,
                                        (uint32_t)prm.py);
      for (int d = 0; d < prm.TD; ++d)
        for (int h = 0; h < prm.TH; h += 2)
          for (int w8 = 0; w8 < prm.TW; w8 += 8) {
            const uint32_t ycell = (uint32_t)((d * prm.TH + h) * prm.TW + w8);
            const uint32_t xcell = (uint32_t)(d * P * slicec + h * prm.HW + w8);
            if (leader) {
              tc_mma_bf16(tmem_base + t * 3 * prm.Cout, adesc0 + xcell + (uint32_t)(t * prm.HW), bdesc0 + ycell, idesc, acc);
              // pointwise conv: rows kd = 1 of the centre (kh = 1) A operand are x[u] itself
              if (prm.dw2 != nullptr && t == 1)
                tc_mma_bf16(tmem_base + 9 * prm.Cout, adesc0 + xcell + (uint32_t)prm.HW, bdesc2 + ycell, idesc2, acc);
            }
            acc = 1;
          }
      if (leader) tc_commit(smem_u32(&empty[s]));
      __syncwarp();
      if (++s == prm.nstages) { s = 0; ph ^= 1; }
    }
    if (leader) tc_commit(smem_u32(done));
    __syncwarp();
  } else if (warp >= 4) {
    // final reduction: accumulator row r = kd * 8P + (ci - cbase) lives in TMEM lane r (M = 128) or lane
    // 32 * (r / 16) + r % 16 (M = 64): either way warp q reads depth tap q, lane = channel
    const int q = warp - 4;
    const int kd = q;
    mbar_wait(smem_u32(done), 0);
    tc_fence_after();
    const bool live = blockIdx.x < prm.ntiles && q < 3;
    // the (kd, tap) block of dw — rows ci of this tile x Cout — is contiguous: stage the warp's 32 rows through shared
    // memory (the stage buffers are free once `done` fired) and add it with 16-byte vector reductions, consecutive lanes
    // on consecutive addresses (row-per-lane scalar atomics are 32 sectors per instruction, 8 P Cout of them per tap);
    // the CTAs start at different taps so that they do not queue on the same addresses
    const int pitch = prm.Cout + 4;
    float* stg = reinterpret_cast<float*>(smem) + q * 32 * pitch;
    const int n4 = 8 * P * prm.Cout / 4;
#pragma unroll 1
    for (int tt = 0; tt < 9 + (prm.dw2 != nullptr ? 1 : 0); ++tt) {
      const int t = tt < 9 ? (tt + (int)blockIdx.x) % 9 : 9;        // 9: the pointwise accumulator (rows kd = 1 only)
      for (int j = 0; j < prm.Cout; j += 16) {
        float v[16];
        tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + t * prm.Cout + j, v);
#pragma unroll
        for (int i = 0; i < 16; i += 4)
          *reinterpret_cast<float4*>(stg + lane * pitch + j + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
      }
      __syncwarp();
      if (live && (t < 9 || kd == 1)) {
        float4* blk = reinterpret_cast<float4*>(
            t < 9 ? prm.dw + ((size_t)(kd * 9 + t) * prm.Cin + cbase) * prm.Cout : prm.dw2 + (size_t)cbase * prm.Cout);
        for (int e = lane; e < n4; e += 32) {
          const int r = (e * 4) / prm.Cout, c = (e * 4) % prm.Cout;
          atomicAdd(blk + e, *reinterpret_cast<const float4*>(stg + r * pitch + c));
        }
      }
      __syncwarp();
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

bool tc_wgrad_kdf_supported(const WgradGeom& wg, const WgP16* p16) {
  if (p16 == nullptr) return false;
  // Cin = 16: M = 64 with 48 real rows (in place of the TS-mode kernel); Cin = 64 / 96 / 128: one CTA row per
  // 32-channel tile
  const bool cin_ok = wg.nA == 16 || (wg.nA % 32 == 0 && wg.nA <= 128);
  if (!(wg.k == 3 && wg.s == 1 && cin_ok && (wg.nB == 16 || wg.nB == 32))) return false;
  if (wg.Ws % 8 != 0 || wg.Hs % 2 != 0) return false;
  for (int i = 0; i < p16->n; ++i)
    if (p16->C[i] % 8 != 0) return false;
  return p16->big_bf16 && p16->small_bf16;
}

int launch_conv_wgrad_kdf(const WgradGeom& wg, float* dw, cudaStream_t s, const WgP16& p16, const void* dres,
                          float* dw2) {
  B3D_REQUIRE(tc_wgrad_kdf_supported(wg, &p16), B3D_ERR_UNSUPPORTED, "wgrad (kd in M): shape not supported");
  B3D_REQUIRE(((uintptr_t)dw & 15) == 0, B3D_ERR_LAYOUT, "wgrad: alignment");
  const int Cin = wg.nA, Cout = wg.nB, P = Cin == 16 ? 2 : 4, nmt = Cin / (8 * P);
  static const int cand[][3] = {{1, 4, 8}, {2, 4, 8}, {2, 4, 16}, {2, 8, 16}, {3, 8, 16}, {4, 8, 16}, {4, 8, 32}};
  KdfParams p;
  memset(&p, 0, sizeof(p));
  const int budget = kWgSmem - 128;
  bool found = false;
  for (int i = 0; i < (int)(sizeof(cand) / sizeof(cand[0])); ++i) {
    const int TD = cand[i][0], TH = cand[i][1], TW = cand[i][2];
    if (found && (TD > wg.Ds * 2 || TH > wg.Hs * 2 || TW > wg.Ws * 2)) continue;
    const int HD = TD + 2, HH = TH + 2, HW = TW;      // no w halo: the kw shifts are in the dy copies
    if (4 * HW > 256) continue;
    const int pslice = ((HH * HW * 16 + 127) / 128) * 128;
    // the A operand spans 16 M groups (M = 128) from the LAST depth slice a K step starts in: 12 are real, the rest
    // must still lie inside this stage's x region or the dy tile (never past the allocation): keep 4 slices of slack
    const long long xbytes = (((long long)HD * P * pslice + 127) / 128) * 128;
    const int py = TD * TH * TW * 16;
    const long long stage = ((xbytes + (dw2 != nullptr ? 4LL : 3LL) * (Cout / 8) * py + 127) / 128) * 128;
    for (int ns = 4; ns >= 2; --ns) {
      const long long last = (long long)(ns - 1) * stage;
      // last K step of the last stage: group 15 starts at (TD-1)*4 slices + 15 slices + h/w offset
      if (ns * stage <= budget && last + ((long long)(TD - 1) * P + 4 * P + 1) * pslice <= budget) {
        p.TD = TD; p.TH = TH; p.TW = TW; p.HD = HD; p.HH = HH; p.HW = HW;
        p.pslice = pslice; p.py = py; p.xbytes = (int)xbytes; p.stage_bytes = (int)stage; p.nstages = ns;
        found = true;
        break;
      }
    }
  }
  B3D_REQUIRE(found, B3D_ERR_UNSUPPORTED, "wgrad (kd in M): no tile fits shared memory (Cin=%d Cout=%d)", Cin, Cout);
  p.dw = dw; p.dw2 = dw2; p.Cin = Cin; p.Cout = Cout; p.P = P;
  B3D_REQUIRE((dw2 == nullptr) == (dres == nullptr) && (dw2 == nullptr || ((uintptr_t)dw2 & 15) == 0),
              B3D_ERR_ARG, "wgrad (kd in M): pointwise operands");
  p.ntd = (wg.Ds + p.TD - 1) / p.TD; p.nth = (wg.Hs + p.TH - 1) / p.TH; p.ntw = (wg.Ws + p.TW - 1) / p.TW;
  p.ntiles = wg.B * p.ntd * p.nth * p.ntw;
  int nsplit = sm_count() / nmt;
  if (nsplit < 1) nsplit = 1;
  if (nsplit > p.ntiles) nsplit = p.ntiles;
  p.nsplit = nsplit;
  WgMaps maps;
  memset(&maps, 0, sizeof(maps));
  p.nsrc = p16.n;
  {
    int g = P;                               // planes per x box: the gcd of the tile and every source's plane count
    for (int i = 0; i < p16.n; ++i) {
      int a = g, b = p16.C[i] / 8;
      while (b) { const int t = a % b; a = b; b = t; }
      g = a;
    }
    p.g = g; p.xbd = g == P ? p.HD : 1;
  }
  int cum = 0;
  for (int i = 0; i < p16.n; ++i) {
    cum += p16.C[i] / 8;
    p.cend8[i] = cum;
    B3D_TRY(make_p16_map_perm(&maps.x[i], p16.big[i], 0, wg.B, wg.Db, wg.Hb, wg.Wb, p16.C[i] / 8, p.HW, p.g, p.HH, p.xbd));
  }
  B3D_REQUIRE(cum * 8 == Cin, B3D_ERR_SHAPE, "wgrad (kd in M): sources hold %d channels, expected %d", cum * 8, Cin);
  B3D_TRY(make_p16_map_perm(&maps.y, p16.small, 1, wg.B, wg.Ds, wg.Hs, wg.Ws, Cout / 8, p.TW, Cout / 8, p.TH, p.TD));
  B3D_TRY(cuda_ok(cudaMemsetAsync(dw, 0, sizeof(float) * 27 * (size_t)Cin * Cout, s), "memset dw"));
  if (dw2 != nullptr) {
    B3D_TRY(make_p16_map_perm(&maps.y2, dres, 1, wg.B, wg.Ds, wg.Hs, wg.Ws, Cout / 8, p.TW, Cout / 8, p.TH, p.TD));
    B3D_TRY(cuda_ok(cudaMemsetAsync(dw2, 0, sizeof(float) * (size_t)Cin * Cout, s), "memset dw (pointwise)"));
  }
  static bool attr = false;
  if (!attr) {
    B3D_TRY(cuda_ok(cudaFuncSetAttribute(conv3_wgrad_kdf_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kWgSmem),
                    "cudaFuncSetAttribute(wgrad_kdf)"));
    attr = true;
  }
  conv3_wgrad_kdf_kernel<<<dim3((unsigned)nsplit, (unsigned)nmt), 256, kWgSmem, s>>>(maps, p);
  B3D_LAUNCH_CHECK("conv3_wgrad_kdf");
  return B3D_OK;
}

// ---- fp32 -> bf16 copies for the tensor-core weight gradient (+ optional column sums = bias gradient)
// thread -> (voxel, channel octet); the octet of a thread is loop-invariant (blockDim % (C/8) == 0)
__global__ void cast_bf16_kernel(const float* __restrict__ src, uint4* __restrict__ dst, long long nvox, int C,
                                 float* __restrict__ colsum) {
  extern __shared__ float sm[];
  const int oc = C / 8;
  const int o = threadIdx.x % oc, vl = threadIdx.x / oc, vpb = blockDim.x / oc;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (long long v = (long long)blockIdx.x * vpb + vl; v < nvox; v += (long long)gridDim.x * vpb) {
    const float4 a = ld_stream(reinterpret_cast<const float4*>(src + v * C + o * 8));
    const float4 b = ld_stream(reinterpret_cast<const float4*>(src + v * C + o * 8) + 1);
    uint4 r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.x) : "f"(a.y), "f"(a.x));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.y) : "f"(a.w), "f"(a.z));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.z) : "f"(b.y), "f"(b.x));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r.w) : "f"(b.w), "f"(b.z));
    dst[v * oc + o] = r;
    acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
    acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
  }
  if (colsum != nullptr) {
    for (int i = threadIdx.x; i < C; i += blockDim.x) sm[i] = 0.f;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(&sm[o * 8 + i], acc[i]);
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(&colsum[i], sm[i]);
  }
}

// space-to-depth variant: dst [B, D, H, W, (parity, C)] bf16  <-  src [B, 2D, 2H, 2W, C] fp32 (channel pitch `pitch`);
// thread -> one 8-channel cell of dst, the channel octet of a thread is loop-invariant
__global__ void cast_bf16_s2d_kernel(const float* __restrict__ src, uint4* __restrict__ dst, int B, int D, int H, int W,
                                     int C, long long pitch, float* __restrict__ colsum) {
  extern __shared__ float sm[];
  const int oc = C / 8;
  const long long total = (long long)B * D * H * W * 8 * oc;
  const int o = threadIdx.x % oc;
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    long long r = i / oc;
    const int par = (int)(r % 8); r /= 8;
    const int w = (int)(r % W); r /= W;
    const int h = (int)(r % H); r /= H;
    const int d = (int)(r % D); r /= D;
    const long long vox = (((r * 2 * D + 2 * d + (par >> 2)) * 2 * H + 2 * h + ((par >> 1) & 1)) * 2 * W) + 2 * w +
                          (par & 1);
    const float4 a = ld_stream(reinterpret_cast<const float4*>(src + vox * pitch + o * 8));
    const float4 b = ld_stream(reinterpret_cast<const float4*>(src + vox * pitch + o * 8) + 1);
    uint4 q;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.x) : "f"(a.y), "f"(a.x));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.y) : "f"(a.w), "f"(a.z));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.z) : "f"(b.y), "f"(b.x));
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(q.w) : "f"(b.w), "f"(b.z));
    dst[i] = q;
    acc[0] += a.x; acc[1] += a.y; acc[2] += a.z; acc[3] += a.w;
    acc[4] += b.x; acc[5] += b.y; acc[6] += b.z; acc[7] += b.w;
  }
  if (colsum != nullptr) {
    for (int i = threadIdx.x; i < C; i += blockDim.x) sm[i] = 0.f;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) atomicAdd(&sm[o * 8 + i], acc[i]);
    __syncthreads();
    for (int i = threadIdx.x; i < C; i += blockDim.x) atomicAdd(&colsum[i], sm[i]);
  }
}

int launch_cast_bf16_s2d(const float* src, void* dst, int B, int D, int H, int W, int C, long long pitch,
                         float* colsum, cudaStream_t s) {
  B3D_REQUIRE(C % 8 == 0 && C <= 2048, B3D_ERR_UNSUPPORTED, "cast_bf16_s2d: channels must be a multiple of 8");
  const int oc = C / 8;
  const int threads = oc >= 256 ? oc : (256 / oc) * oc;
  const long long total = (long long)B * D * H * W * 8 * oc;
  long long blocks = (total + (long long)threads * 8 - 1) / ((long long)threads * 8);
  const long long cap = 8LL * sm_count();
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (colsum != nullptr) B3D_TRY(cuda_ok(cudaMemsetAsync(colsum, 0, sizeof(float) * C, s), "memset colsum"));
  cast_bf16_s2d_kernel<<<(unsigned)blocks, threads, sizeof(float) * C, s>>>(src, (uint4*)dst, B, D, H, W, C, pitch,
                                                                            colsum);
  B3D_LAUNCH_CHECK("cast_bf16_s2d");
  return B3D_OK;
}

// "tap-stacked" bf16 copy of a NARROW tensor (Cn < 8 channels: the 2-channel input volume, the 2-3 channel
// gradients of the output convs):  dst[v][(t, c)] = src[v + sgn*(t - pad)][c]  for the k^3 taps t, zero outside the
// volume and in the padding up to nA = 8*ceil(k^3*Cn/8) channels.  The weight gradient of such a layer is then ONE
// K = voxels GEMM (the KS = 1 case of conv3_wgrad_tc_kernel) with all taps in the M dimension instead of k^3 MMAs
// whose M = 128 rows hold 2 real channels.  sgn = +1 stacks the layer input x (rows (t, ci)); sgn = -1 stacks dy
// (dw[t][ci][co] = sum_u x[u][ci] dy[u - (t - pad)][co], rows (t, co)).  thread -> one 16-byte cell.
constexpr int kStD = 4, kStH = 8, kStW = 32;     // voxel tile of the stacking kernel
__global__ void __launch_bounds__(256)
    cast_stack_bf16_kernel(const float* __restrict__ src, uint4* __restrict__ dst, int B, int D, int H, int W, int Cn,
                           long long pitch, int k, int sgn, int nA, int ntd, int nth, int ntw) {
  extern __shared__ float sh[];                  // halo tile [kStD+2p][kStH+2p][kStW+2p][Cn], zero outside the volume
  __shared__ int lut[256];                       // stacked row -> offset inside the halo tile (-1: zero padding)
  const int cells = nA / 8, pad = k / 2, rows = k * k * k * Cn;
  const int ED = kStD + 2 * pad, EH = kStH + 2 * pad, EW = kStW + 2 * pad;
  const int ntiles = B * ntd * nth * ntw;
  for (int row = threadIdx.x; row < nA; row += 256) {
    int off = INT_MIN;
    if (row < rows) {
      const int t = row / Cn, c = row - t * Cn;
      const int od = sgn * (t / (k * k) - pad), oh = sgn * ((t / k) % k - pad), ow = sgn * (t % k - pad);
      off = ((od * EH + oh) * EW + ow) * Cn + c;
    }
    lut[row] = off;
  }
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    int q = tile;
    const int wt = q % ntw; q /= ntw;
    const int ht = q % nth; q /= nth;
    const int dt = q % ntd; q /= ntd;
    const int b = q, d0 = dt * kStD, h0 = ht * kStH, w0 = wt * kStW;
    __syncthreads();
    for (int i = threadIdx.x; i < ED * EH * EW * Cn; i += 256) {
      const int c = i % Cn; int r = i / Cn;
      const int ew = r % EW; r /= EW;
      const int eh = r % EH; const int ed = r / EH;
      const int dd = d0 + ed - pad, hh = h0 + eh - pad, ww = w0 + ew - pad;
      float v = 0.f;
      if (dd >= 0 && dd < D && hh >= 0 && hh < H && ww >= 0 && ww < W)
        v = __ldg(src + ((((long long)b * D + dd) * H + hh) * W + ww) * pitch + c);
      sh[i] = v;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < kStD * kStH * kStW * cells; i += 256) {
      const int cell = i % cells; int r = i / cells;
      const int lw = r % kStW; r /= kStW;
      const int lh = r % kStH; const int ld = r / kStH;
      const int d = d0 + ld, h = h0 + lh, w = w0 + lw;
      if (d >= D || h >= H || w >= W) continue;
      const int base = (((ld + pad) * EH + (lh + pad)) * EW + (lw + pad)) * Cn;
      float v[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int off = lut[cell * 8 + e];
        v[e] = off == INT_MIN ? 0.f : sh[base + off];
      }
      uint4 o;
      asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(o.x) : "f"(v[1]), "f"(v[0]));
      asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(o.y) : "f"(v[3]), "f"(v[2]));
      asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(o.z) : "f"(v[5]), "f"(v[4]));
      asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(o.w) : "f"(v[7]), "f"(v[6]));
      dst[((((long long)b * D + d) * H + h) * W + w) * cells + cell] = o;
    }
  }
}

int launch_cast_stack_bf16(const float* src, void* dst, int B, int D, int H, int W, int Cn, long long pitch, int k,
                           int sgn, int nA, cudaStream_t s) {
  B3D_REQUIRE(Cn >= 1 && Cn < 8 && nA % 8 == 0 && nA <= 256, B3D_ERR_UNSUPPORTED,
              "cast_stack: narrow tensors only (1..7 channels)");
  const int pad = k / 2;
  const size_t smem = sizeof(float) * (size_t)(kStD + 2 * pad) * (kStH + 2 * pad) * (kStW + 2 * pad) * Cn;
  static bool attr = false;
  if (!attr) {
    B3D_TRY(cuda_ok(cudaFuncSetAttribute(cast_stack_bf16_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024),
                    "cudaFuncSetAttribute(cast_stack)"));
    attr = true;
  }
  const int ntd = (D + kStD - 1) / kStD, nth = (H + kStH - 1) / kStH, ntw = (W + kStW - 1) / kStW;
  const long long ntiles = (long long)B * ntd * nth * ntw;
  const long long cap = 4LL * sm_count();
  cast_stack_bf16_kernel<<<(unsigned)(ntiles < cap ? ntiles : cap), 256, smem, s>>>(src, (uint4*)dst, B, D, H, W, Cn,
                                                                                   pitch, k, sgn, nA, ntd, nth, ntw);
  B3D_LAUNCH_CHECK("cast_stack_bf16");
  return B3D_OK;
}

int launch_cast_bf16(const float* src, void* dst, long long nvox, int C, float* colsum, cudaStream_t s) {
  B3D_REQUIRE(C % 8 == 0 && C <= 2048, B3D_ERR_UNSUPPORTED, "cast_bf16: channels must be a multiple of 8");
  const int oc = C / 8;
  const int threads = oc >= 256 ? oc : (256 / oc) * oc;
  const int vpb = threads / oc;
  long long blocks = (nvox + (long long)vpb * 8 - 1) / ((long long)vpb * 8);
  const long long cap = 8LL * sm_count();
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  if (colsum != nullptr) B3D_TRY(cuda_ok(cudaMemsetAsync(colsum, 0, sizeof(float) * C, s), "memset colsum"));
  cast_bf16_kernel<<<(unsigned)blocks, threads, sizeof(float) * C, s>>>(src, (uint4*)dst, nvox, C, colsum);
  B3D_LAUNCH_CHECK("cast_bf16");
  return B3D_OK;
}

}  // namespace b3d
