// b3d — stride-1 SAME convolutions (3x3x3 and 1x1x1) as implicit GEMMs on the 5th-gen tensor cores
// (tcgen05.mma, accumulators in TMEM).  Used for Conv3D forward (reference layers/resnet.py:30-37,
// 80-87,96-103) and, with flipped/transposed packed weights, for its data gradient.
//
// "Shifted GEMM on a resident halo tile":
//   * a CTA owns an output tile of TD x 16 x (8*NW) voxels.  For each chunk of CK input channels
//     (16 as bf16 / 8 as tf32 = one MMA K step) eight LOADER warps read the (TD+2) x 18 x (8*NW+2)
//     halo of the fp32 NDHWC activation ONCE with 128-bit loads (zero outside the volume = TF 'SAME'
//     padding), convert it to the operand type in registers, and store it to shared memory as two
//     channel planes  plane[d'][h'][w'] of 16-byte cells — the canonical K-major SWIZZLE_NONE UMMA
//     layout with a 16-byte row pitch, so that ANY voxel shift is just a start-address offset.
//     (Round-1a used TMA with 16-byte boxes for this; ncu showed ~3 cycles per cell, i.e. the kernel
//     was TMA-issue-bound; a thread loader is faster and converts to bf16 for free.)
//   * every tap is then an MMA whose A descriptor points into that same halo at the tap's offset:
//     M = 128 rows = a 16(h) x 8(w) patch (8 consecutive w = one core matrix, SBO = one halo row),
//     K = CK channels (LBO = one plane), N = Cout.  No im2col, no re-load per tap.
//   * weights are pre-packed (bf16 / tf32-rounded) into the matching B layout and streamed one kd slab
//     (9 taps) at a time through a 3-deep ring with bulk copies (cp.async.bulk + mbarrier complete_tx).
//   * warp-specialised, persistent: warps 0-3 = epilogue (tcgen05.ld -> +bias -> NDHWC store, fused
//     GroupNorm chunk statistics or global-average-pool sums), warps 4-11 = loaders, warp 12 = single
//     thread MMA issuer, warp 13 = weight producer (+TMEM alloc); 2 TMEM accumulator stages overlap
//     epilogue(i) with MMA(i+1).
//
// "kd-folded" variant (TcCfg::FOLD, 3x3x3, Cout tile 16 | 32): the cost of a small-N SS-mode tcgen05.mma is the fetch
// of its 4 KB A tile from shared memory (~40-56 cycles whatever N is, profiles/r01_umma_rate.txt), so the narrow
// layers are bound by the NUMBER of MMAs.  Folding the depth taps into N cuts that number 2-2.4x: for every INPUT
// depth slice z of the halo and every (kh, kw), ONE MMA multiplies the slice's patch with [W(kd=2) | W(kd=1) | W(kd=0)]
// (N' = 3N columns), and its D block lands on the accumulators of the three OUTPUT slices z-2, z-1, z (relative to the
// halo), which are adjacent column blocks in TMEM:  9 (TD+2) MMAs per chunk and patch column instead of 27 TD.
// Accumulator blocks are first touched by the kd = 0 column block of the first (chunk, kh, kw) step — issued as its
// own N-wide MMA with accumulate = 0 next to a 2N-wide one for the other two blocks; two blocks at either end of the
// TMEM column range receive the out-of-tile contributions and are never read.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "conv_common.cuh"
#include "tc_ptx.cuh"

namespace b3d {

// ------------------------------------------------------------------------------------------ config
template <int N_, int TD_, int NW_, int KS_, int HB_, int OP_, int FOLD_ = 0>
struct TcCfg {
  static constexpr int N = N_, TD = TD_, NW = NW_, KS = KS_;
  static constexpr bool FOLD = FOLD_ != 0;            // depth taps folded into N (see the header comment)
  static constexpr int NB = FOLD ? 3 * N : N;         // rows of one B tile = N of one (unsplit) MMA
  static constexpr int HB = HB_;                      // halo before the tile: tap k reads offset k - HB
  static constexpr int OP = OP_;                      // operand type: OP_TF32 | OP_BF16 | OP_F16
  static constexpr bool BF16 = OP_ != OP_TF32;        // 16-bit operands (bf16 or fp16): 8 channels per cell
  static constexpr int T = BF16 ? 8 : 4;              // channels per 16-byte cell
  static constexpr int CK = 2 * T;                    // channels per chunk = one MMA K step
  static constexpr int TAPS = KS * KS * KS;
  static constexpr int TH = 16, TW = 8 * NW, P = TD * NW;
  static constexpr int HD = TD + KS - 1, HH = TH + KS - 1, HW = TW + KS - 1;
  static constexpr int NVC = HD * HH * HW;            // halo voxels (cells per plane)
  // halo stage in shared memory: [HD][HH][2 planes][HW] 16-byte cells — the two channel octets of a K chunk sit side
  // by side inside every (d, h) row, which is exactly what ONE 5-D TMA box {8*HW, 2, HH, HD, 1} of a P16 operand
  // delivers; the thread loader writes the same layout.  UMMA: LBO (K direction = plane) = HW cells, SBO (next 8-row
  // group = next h row) = RP cells; a tap (kd, kh, kw) is a start-address offset of ((kd*HH + kh)*RP + kw) cells.
  static constexpr int RP = 2 * HW;                   // row pitch in cells
  static constexpr int HALO_TX = HD * HH * RP * 16;   // bytes one TMA box writes
  static constexpr int HALO_BYTES = ((HALO_TX + 127) / 128) * 128;
  static constexpr int TAP_BYTES = 2 * N * 16;        // B tile of one tap: 2 planes x N rows x 16 B
  static constexpr int TPS = KS * KS;                 // taps per weight stage (one kd slab; 1 for 1x1x1;
                                                      // FOLD: one kh row = 3 (kh, kw) tiles of 3N rows)
  static constexpr int WST_BYTES = TPS * TAP_BYTES;
  static constexpr int WS = (KS == 1) ? 8 : 3;
  static constexpr int ACC_COLS = 256;                // per accumulator stage (P*N <= 256)
  static constexpr int BAR_BYTES = 768;               // mbarriers + TMEM slot (256 B) | CTA-level statistics / pooling sums
  static constexpr int HS = (3 * HALO_BYTES + WS * WST_BYTES + BAR_BYTES <= 220 * 1024) ? 3 : 2;
  static constexpr int SMEM = HS * HALO_BYTES + WS * WST_BYTES + BAR_BYTES;
  static constexpr int ACC_BLOCKS = FOLD ? NW * (TD + 4) : P;     // N-column accumulator blocks per stage
  static_assert(ACC_BLOCKS * N <= ACC_COLS, "accumulators exceed a TMEM stage");
  static_assert(!FOLD || (KS == 3 && HB == 1 && BF16 && (N == 16 || N == 32)), "kd-folded variant: 3x3x3, 16-bit, N 16|32");
  // TMEM column block of output patch (pd, pw) within a stage
  static constexpr __host__ __device__ int acc_block(int pd, int pw) { return FOLD ? pw * (TD + 4) + pd + 2 : pd * NW + pw; }
  static_assert(SMEM <= 227 * 1024, "shared memory budget");
};

struct TcParams {
  const float* x;      // fp32 NDHWC input, channel pitch xp
  const void* wp;      // packed weights [nsplit][chunk][tap][2 planes][N][T]
  const float* bias;   // nullable
  float* y;
  double* stats;       // nullable: GroupNorm chunk (sum, sum^2) of y
  float* gap;          // nullable: per-(b, channel) sums of y
  int B, D, H, W, Cin, Cout;
  long long xp, yp;    // channel pitches
  int ntd, nth, ntw, ntiles;
  int accumulate, groups;
  long long vpc;       // voxels per GN chunk (of the tensor y is stored as)
  long long voff;      // first voxel of y inside the whole volume (depth slabs; 0 otherwise)
  // centre-tap K segment (3x3x3 only): K chunks >= `cfull` are multiplied with the 1x1x1 operand `wpc` (packed like a
  // k = 1 layer: [nsplit][chunk][1 tap][2 planes][N][T]) at the centre tap only — the data gradient of a ResnetBlock's
  // pointwise conv computed inside the data gradient of its first 3x3x3 conv (both are gradients w.r.t. the block
  // input: one kernel, one output, no add).  cfull = all chunks: no such segment.
  int cfull;
  const void* wpc;
  // output split into up to 4 compact tensors by channel ranges (stride-1 convs; nyd = 0: y / yp)
  int nyd, yde[4];
  float* yd[4];
  // stride-2 family (conv_s2.cu): the kernel works on the COARSE grid [D,H,W];
  //   s2d: x is the fine tensor [B,2D,2H,2W,Csub]; virtual input channel k' = parity*Csub + c  (space-to-depth)
  //   d2s: y is the fine tensor [B,2D,2H,2W,Csub]; virtual output column n' = parity*Csub + c (depth-to-space)
  int s2d, d2s, Csub;
  // slab halos (whole-volume inference sharded along D): x holds Din depth slices (its own units: fine for s2d) and
  // logical slice i lives at buffer slice i + doff; slices outside [0, Din) read as zero
  int Din, doff;
  // channel padding: Cin / Cout above are the padded (virtual) counts the MMAs run on; the tensors hold cin_real /
  // cout_real channels (first conv: 2 input channels; output convs: 2-3 classes).  act: 1 = sigmoid epilogue.
  int cin_real, cout_real, act;
  // split-K (small volumes with long reductions: far fewer tiles than SMs): blockIdx.z owns `kchunks` consecutive K
  // chunks and stores its partial result into slice z of a workspace (`y` points at it, `ws_slice` elements per
  // slice); conv_finish_kernel then sums the slices and applies bias / statistics / GAP
  int ksplit, kchunks;
  long long ws_slice;
  // P16 input operand (16-bit [B, D, H, C/8, W, 8] twins, see common.cuh): x16 = 1 -> `src` holds up to 4 source
  // tensors whose channels are concatenated virtually (K chunk -> source by `cend`, the cumulative channel ends);
  // tma = 1 -> the halo of a chunk is fetched by one TMA box from the source's tensor map (stride-1 addressing),
  // otherwise (space-to-depth addressing of the stride-2 family) by the loader warps with 16-byte loads.
  int x16, tma, nsrc;
  const void* src[4];
  int cend[4];         // cumulative channel count after source i (of the concatenated input)
  int sc8[4];          // channel octets (planes) of source i
};

struct alignas(64) TcMaps {
  CUtensorMap m[4];
};

__device__ __forceinline__ void tc_mma_f16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
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

// 256-bit streaming load (one full 32-byte sector per lane; sm_100 LDG.E.256)
__device__ __forceinline__ void ld256(const float* p, float* r) {
  asm volatile("ld.global.nc.L1::no_allocate.v8.f32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
               : "=f"(r[0]), "=f"(r[1]), "=f"(r[2]), "=f"(r[3]), "=f"(r[4]), "=f"(r[5]), "=f"(r[6]), "=f"(r[7])
               : "l"(p));
}

// 256-bit store: one full 32-byte sector per lane (sm_100 STG.E.256).  The epilogue's lanes each own the 16 channels
// (64 bytes) of one voxel; with 128-bit stores every warp instruction touches 32 sectors HALF — twice the L2 write
// requests, all of them partial
__device__ __forceinline__ void st256(float* p, float a, float b, float c, float d, float e, float f, float g, float h) {
  asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "f"(e),
               "f"(f), "f"(g), "f"(h)
               : "memory");
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
  return r;
}

__device__ __forceinline__ uint32_t pack_f16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));   // saturate: no inf operands
  return r;
}
template <int OP>
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  return OP == OP_F16 ? pack_f16x2(lo, hi) : pack_bf16x2(lo, hi);
}

// add a warp's running GroupNorm sums to stats[chunk]: one pair of fp64 atomics per warp when all its lanes are in the
// same chunk (the common case), per lane otherwise.  Must be called by all 32 lanes.
__device__ __noinline__ void flush_stats(double* stats, int cur_chunk, float s0, float s1, int lane) {
  const int cc = __reduce_max_sync(0xffffffffu, cur_chunk);
  if (cc < 0) return;                                               // nothing accumulated anywhere in the warp
  const bool uni = __all_sync(0xffffffffu, cur_chunk == cc || cur_chunk < 0);
  if (uni) {
    const float a0 = warp_sum(cur_chunk >= 0 ? s0 : 0.f), a1 = warp_sum(cur_chunk >= 0 ? s1 : 0.f);
    if (lane == 0) {
      atomicAdd(&stats[2 * cc], (double)a0);
      atomicAdd(&stats[2 * cc + 1], (double)a1);
    }
  } else if (cur_chunk >= 0) {
    atomicAdd(&stats[2 * cur_chunk], (double)s0);
    atomicAdd(&stats[2 * cur_chunk + 1], (double)s1);
  }
}

// the same for a warp's LAST flush: warps of a CTA end in the same chunk (or two), so their sums are combined in shared
// memory (4 slots tagged with the chunk; a slot taken by another chunk falls back to the global atomics) and written
// by the CTA once, after its final barrier
__device__ __noinline__ void flush_stats_cta(double* stats, int cur_chunk, float s0, float s1, int lane, double* acc,
                                             int* tag) {
  const int cc = __reduce_max_sync(0xffffffffu, cur_chunk);
  if (cc < 0) return;
  const bool uni = __all_sync(0xffffffffu, cur_chunk == cc || cur_chunk < 0);
  if (uni) {
    const float a0 = warp_sum(cur_chunk >= 0 ? s0 : 0.f), a1 = warp_sum(cur_chunk >= 0 ? s1 : 0.f);
    if (lane == 0) {
      const int slot = cc & 3;
      const int old = atomicCAS(&tag[slot], -1, cc);
      if (old == -1 || old == cc) {
        atomicAdd(&acc[2 * slot], (double)a0);
        atomicAdd(&acc[2 * slot + 1], (double)a1);
      } else {
        atomicAdd(&stats[2 * cc], (double)a0);
        atomicAdd(&stats[2 * cc + 1], (double)a1);
      }
    }
  } else if (cur_chunk >= 0) {
    atomicAdd(&stats[2 * cur_chunk], (double)s0);
    atomicAdd(&stats[2 * cur_chunk + 1], (double)s1);
  }
}

// Column sums over the 32 lanes of 16 per-lane values by a butterfly reduce-scatter: 15 + 1 shuffles instead of 16 warp
// sums (80).  Afterwards every lane holds the total of ONE column: column = (lane >> 1) with its 4 bits reversed... see
// `col` below; lanes 2k and 2k + 1 hold the same column.
__device__ __forceinline__ float warp_colsum16(const float (&v)[16], int lane, int& col) {
  float a[8], b[4], c[2];
  const bool h16 = lane & 16, h8 = lane & 8, h4 = lane & 4, h2 = lane & 2;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float keep = h16 ? v[i + 8] : v[i], send = h16 ? v[i] : v[i + 8];
    a[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);              // column i + 8 * bit4
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float keep = h8 ? a[i + 4] : a[i], send = h8 ? a[i] : a[i + 4];
    b[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);               // column i + 4 * bit3 + 8 * bit4
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float keep = h4 ? b[i + 2] : b[i], send = h4 ? b[i] : b[i + 2];
    c[i] = keep + __shfl_xor_sync(0xffffffffu, send, 4);               // column i + 2 * bit2 + 4 * bit3 + 8 * bit4
  }
  const float keep = h2 ? c[1] : c[0], send = h2 ? c[0] : c[1];
  float d = keep + __shfl_xor_sync(0xffffffffu, send, 2);              // column bit1 + 2 * bit2 + 4 * bit3 + 8 * bit4
  d += __shfl_xor_sync(0xffffffffu, d, 1);
  col = (h2 ? 1 : 0) | (h4 ? 2 : 0) | (h8 ? 4 : 0) | (h16 ? 8 : 0);
  return d;
}

constexpr int kLoaderWarps = 8;
// Number of MMA-issuing warps (each owns the patches p = its index mod kMmaWarps).  One warp can issue a tcgen05.mma
// only every ~50 cycles (profiles/r01_umma_rate.txt), but measured with 2 issuers this kernel does not get faster (the
// shifted-tile A fetch from shared memory, ~56 cycles per N = 16 MMA here, is the limit, not the issue rate): 1.
constexpr int kMmaWarps = 1;
static_assert(kMmaWarps == 1, "warp roles below assume one MMA-issuing warp");
// warps: 0-3 epilogue | 4-11 operand loaders (thread-loader form) or 8 MORE epilogue warps (TMA form: the loaders have
// nothing to do, and the 1x1x1 / narrow layers are bound by the epilogue's store rate: profiles/r02e) | 12 MMA issuer |
// 13 weight producer (+ TMEM alloc) | 14 TMA producer of the operand halos
constexpr int kTmaWarp = kLoaderWarps + 6;
constexpr int kTcThreads = (kTmaWarp + 1) * 32;

template <class C>
__global__ void __launch_bounds__(kTcThreads, 1) conv_tc_kernel(const TcParams prm, const __grid_constant__ TcMaps maps) {
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* halo = smem;
  uint8_t* wst = smem + C::HS * C::HALO_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(wst + C::WS * C::WST_BYTES);
  uint64_t* halo_full = bars;                  // [HS]  128 loader arrivals
  uint64_t* halo_empty = bars + 4;             // [HS]  tcgen05.commit
  uint64_t* w_full = bars + 8;                 // [WS]  expect_tx + bulk copy
  uint64_t* w_empty = bars + 8 + C::WS;        // [WS]  tcgen05.commit
  uint64_t* acc_full = bars + 8 + 2 * C::WS;   // [2]
  uint64_t* acc_empty = acc_full + 2;          // [2]  4 epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  // final flush of the epilogue warps' running sums goes through shared memory: one set of global atomics per CTA
  double* cta_stat = reinterpret_cast<double*>(reinterpret_cast<uint8_t*>(bars) + 256);   // [4 slots][2]
  int* cta_stat_tag = reinterpret_cast<int*>(cta_stat + 8);                                // [4] chunk of the slot, -1 = free
  float* cta_gap = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 384);       // [64] (N <= 64)
  int* cta_gap_b = reinterpret_cast<int*>(cta_gap + 64);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nchunks_all = prm.Cin / C::CK;
  const int c_begin = blockIdx.z * prm.kchunks;
  const int nchunks = min(prm.kchunks, nchunks_all - c_begin);   // this CTA's K chunks: [c_begin, c_begin + nchunks)
  const int nsp = blockIdx.y;  // N split
  // a persistent CTA owns a CONTIGUOUS range of tiles: its GroupNorm chunk (and sample) then changes once or twice in
  // its life instead of every other tile, which is what the number of same-address statistics atomics scales with
  // (~15 ns each once they queue up on one L2 address)
  const int tpc = prm.ntiles / (int)gridDim.x, trem = prm.ntiles % (int)gridDim.x;
  const int tile0 = (int)blockIdx.x * tpc + min((int)blockIdx.x, trem), tile1 = tile0 + tpc + ((int)blockIdx.x < trem ? 1 : 0);

  if (threadIdx.x == 0) {
    for (int i = 0; i < C::HS; ++i) { mbar_init(smem_u32(&halo_full[i]), prm.tma ? 1 : kLoaderWarps * 32); mbar_init(smem_u32(&halo_empty[i]), kMmaWarps); }
    for (int i = 0; i < C::WS; ++i) { mbar_init(smem_u32(&w_full[i]), 1); mbar_init(smem_u32(&w_empty[i]), kMmaWarps); }
    for (int i = 0; i < 2; ++i) { mbar_init(smem_u32(&acc_full[i]), kMmaWarps); mbar_init(smem_u32(&acc_empty[i]), prm.tma ? 4 + kLoaderWarps : 4); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (threadIdx.x < 64) cta_gap[threadIdx.x] = 0.f;
  if (threadIdx.x < 8) cta_stat[threadIdx.x] = 0.0;
  if (threadIdx.x < 4) cta_stat_tag[threadIdx.x] = -1;
  if (threadIdx.x == 0) *cta_gap_b = -1;
  if (warp == kLoaderWarps + 5) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)),
                 "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_trigger();
  pdl_wait();          // everything above overlaps the tail of the previous kernel

  if (warp == kTmaWarp) {
    // ============ operand loader, TMA form: one elected thread fetches the halo of every K chunk as ONE 5-D box
    // {HW voxels, 2 planes, HH, HD, 1} of the source's P16 tensor map (zero fill outside the volume = TF 'SAME' padding)
    if (prm.tma && lane == 0) {
      int hs = 0, hph = 0;
      for (int tile = tile0; tile < tile1; ++tile) {
        int t = tile;
        const int wt = t % prm.ntw; t /= prm.ntw;
        const int ht = t % prm.nth; t /= prm.nth;
        const int dt = t % prm.ntd; t /= prm.ntd;
        const int b = t;
        const int w0 = wt * C::TW - C::HB, h0 = ht * C::TH - C::HB, d0 = dt * C::TD - C::HB + prm.doff;
        for (int c = 0; c < nchunks; ++c) {
          const int ch0 = (c_begin + c) * C::CK;                 // first channel of the chunk in the concatenated input
          int si = 0;
          while (si + 1 < prm.nsrc && ch0 >= prm.cend[si]) ++si;
          const int pl = (ch0 - (si > 0 ? prm.cend[si - 1] : 0)) >> 3;
          mbar_wait(smem_u32(&halo_empty[hs]), hph ^ 1);
          const uint32_t full = smem_u32(&halo_full[hs]);
          mbar_expect_tx(full, C::HALO_TX);
          tma_load_5d(smem_u32(halo + hs * C::HALO_BYTES), &maps.m[si], 4 * w0, pl, h0, d0, b, full);
          if (++hs == C::HS) { hs = 0; hph ^= 1; }
        }
      }
    }
  } else if (warp >= 4 && warp < 4 + kLoaderWarps && !prm.tma) {
    // ============ operand loaders: global fp32 -> (bf16|tf32) cells in shared memory ============
    const int lw = warp - 4;
    int hs = 0, hph = 0;
    for (int tile = tile0; tile < tile1; ++tile) {
      int t = tile;
      const int wt = t % prm.ntw; t /= prm.ntw;
      const int ht = t % prm.nth; t /= prm.nth;
      const int dt = t % prm.ntd; t /= prm.ntd;
      const int b = t;
      const int w0 = wt * C::TW - C::HB, h0 = ht * C::TH - C::HB, d0 = dt * C::TD - C::HB;
      const float* xb = prm.x + (long long)b * prm.Din * prm.H * prm.W * prm.xp * (prm.s2d ? 4 : 1);
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(smem_u32(&halo_empty[hs]), hph ^ 1);
        uint8_t* dst0 = halo + hs * C::HALO_BYTES;
        const int cg = c_begin + c;              // global K-chunk index
        const float* xc = xb + cg * C::CK;
        int sp_d = 0, sp_h = 0, sp_w = 0;      // s2d: parity of this chunk's channels
        int chv = cg * C::CK;                  // first (virtual) channel of the chunk inside the source tensor(s)
        if (prm.s2d) {
          const int par = (cg * C::CK) / prm.Csub;
          chv = (cg * C::CK) % prm.Csub;
          xc = xb + chv;
          sp_d = par >> 2; sp_h = (par >> 1) & 1; sp_w = par & 1;
        }
        constexpr int kVoxPerPass = kLoaderWarps * 32;
        constexpr int kUnroll = 4;
        if (C::BF16 && prm.x16) {
          // P16 source (16-bit twins, possibly a virtual concat of several tensors): a voxel's chunk is two 16-byte
          // cells one plane (W cells) apart; no conversion
          int si = 0;
          while (si + 1 < prm.nsrc && chv >= prm.cend[si]) ++si;
          const int pl = (chv - (si > 0 ? prm.cend[si - 1] : 0)) >> 3, c8 = prm.sc8[si];
          const int fs = prm.s2d ? 2 : 1;
          const long long Hf = (long long)prm.H * fs, Wf = (long long)prm.W * fs;
          const uint4* xs = reinterpret_cast<const uint4*>(prm.src[si]) + (long long)b * prm.Din * Hf * c8 * Wf;
          for (int v0 = lw * 32 + lane; v0 < C::NVC; v0 += kVoxPerPass * kUnroll) {
            uint4 q[kUnroll][2];
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
              const int v = v0 + u * kVoxPerPass;
              const int cw = v % C::HW, q2 = v / C::HW;
              const int ch = q2 % C::HH, cd = q2 / C::HH;
              const int gd = d0 + cd, gh = h0 + ch, gw = w0 + cw;
              const int bd = (prm.s2d ? 2 * gd + sp_d : gd) + prm.doff;
              const bool ok = v < C::NVC && bd >= 0 && bd < prm.Din && gh >= 0 && gh < prm.H && gw >= 0 && gw < prm.W;
              q[u][0] = q[u][1] = make_uint4(0u, 0u, 0u, 0u);
              if (ok) {
                const long long hh = prm.s2d ? 2 * gh + sp_h : gh, ww = prm.s2d ? 2 * gw + sp_w : gw;
                const uint4* sp = xs + (((long long)bd * Hf + hh) * c8 + pl) * Wf + ww;
                q[u][0] = __ldg(sp);
                q[u][1] = __ldg(sp + Wf);
              }
            }
#pragma unroll
            for (int u = 0; u < kUnroll; ++u) {
              const int v = v0 + u * kVoxPerPass;
              if (v < C::NVC) {
                const int cw = v % C::HW, row = v / C::HW;
                uint8_t* d = dst0 + (row * C::RP + cw) * 16;
                *reinterpret_cast<uint4*>(d) = q[u][0];
                *reinterpret_cast<uint4*>(d + C::HW * 16) = q[u][1];
              }
            }
          }
        } else {
        // one lane = one halo voxel: the whole CK-channel chunk is fetched with 256-bit loads (full 32-byte
        // sectors), converted, and written as one 16-byte cell per plane (a warp stores 512 contiguous bytes)
        constexpr int kRegs = C::BF16 ? 16 : 8;
        for (int v0 = lw * 32 + lane; v0 < C::NVC; v0 += kVoxPerPass * kUnroll) {
          float r[kUnroll][kRegs];
#pragma unroll
          for (int u = 0; u < kUnroll; ++u) {
            const int v = v0 + u * kVoxPerPass;
            const int cw = v % C::HW, q = v / C::HW;
            const int ch = q % C::HH, cd = q / C::HH;
            const int gd = d0 + cd, gh = h0 + ch, gw = w0 + cw;
            const int bd = (prm.s2d ? 2 * gd + sp_d : gd) + prm.doff;      // buffer depth slice
            const bool ok = v < C::NVC && bd >= 0 && bd < prm.Din && gh >= 0 && gh < prm.H && gw >= 0 && gw < prm.W;
#pragma unroll
            for (int i = 0; i < kRegs; ++i) r[u][i] = 0.f;
            if (ok && prm.cin_real < C::CK) {
              // narrow input (fewer real channels than one K step): scalar loads, zero padding stays in r[]
              const float* src = xc + (((long long)bd * prm.H + gh) * prm.W + gw) * prm.xp;
#pragma unroll
              for (int i = 0; i < 8; ++i)
                if (i < prm.cin_real) r[u][i] = __ldg(src + i);
            } else if (ok) {
              const float* src =
                  prm.s2d ? xc + (((long long)bd * (2 * prm.H) + (2 * gh + sp_h)) * (2 * prm.W) + (2 * gw + sp_w)) * prm.xp
                          : xc + (((long long)bd * prm.H + gh) * prm.W + gw) * prm.xp;
              ld256(src, r[u]);
              if (C::BF16) ld256(src + 8, r[u] + 8);
            }
          }
#pragma unroll
          for (int u = 0; u < kUnroll; ++u) {
            const int v = v0 + u * kVoxPerPass;
            if (v < C::NVC) {
              uint4 o0, o1;
              if (C::BF16) {
                o0.x = pack_half2<C::OP>(r[u][0], r[u][1]); o0.y = pack_half2<C::OP>(r[u][2], r[u][3]);
                o0.z = pack_half2<C::OP>(r[u][4], r[u][5]); o0.w = pack_half2<C::OP>(r[u][6], r[u][7]);
                o1.x = pack_half2<C::OP>(r[u][8], r[u][9]); o1.y = pack_half2<C::OP>(r[u][10], r[u][11]);
                o1.z = pack_half2<C::OP>(r[u][12], r[u][13]); o1.w = pack_half2<C::OP>(r[u][14], r[u][15]);
              } else {
                o0.x = __float_as_uint(r[u][0]); o0.y = __float_as_uint(r[u][1]);
                o0.z = __float_as_uint(r[u][2]); o0.w = __float_as_uint(r[u][3]);
                o1.x = __float_as_uint(r[u][4]); o1.y = __float_as_uint(r[u][5]);
                o1.z = __float_as_uint(r[u][6]); o1.w = __float_as_uint(r[u][7]);
              }
              const int cw = v % C::HW, row = v / C::HW;
              uint8_t* d = dst0 + (row * C::RP + cw) * 16;
              *reinterpret_cast<uint4*>(d) = o0;
              *reinterpret_cast<uint4*>(d + C::HW * 16) = o1;
            }
          }
        }
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy stores -> UMMA reads
        mbar_arrive(smem_u32(&halo_full[hs]));
        if (++hs == C::HS) { hs = 0; hph ^= 1; }
      }
    }
  } else if (warp == kLoaderWarps + 5) {
    // ============ weight producer (bulk copies, one kd slab of taps per stage) ============
    if (lane == 0) {
      int ws = 0, wph = 0;
      const uint8_t* wsrc =
          reinterpret_cast<const uint8_t*>(prm.wp) + ((size_t)nsp * prm.cfull + c_begin) * C::TAPS * C::TAP_BYTES;
      constexpr int kStagesPerChunk = C::TAPS / C::TPS;
      const uint8_t* wsrc_c = reinterpret_cast<const uint8_t*>(prm.wpc) +
                              (size_t)nsp * (nchunks_all - prm.cfull) * C::TAP_BYTES;      // centre-tap segment
      for (int tile = tile0; tile < tile1; ++tile) {
        for (int c = 0; c < nchunks; ++c) {
          const int cg = c_begin + c;
          if (cg >= prm.cfull) {          // one stage holding the single tap tile of this chunk
            mbar_wait(smem_u32(&w_empty[ws]), wph ^ 1);
            const uint32_t full = smem_u32(&w_full[ws]);
            mbar_expect_tx(full, C::TAP_BYTES);
            bulk_g2s(smem_u32(wst + ws * C::WST_BYTES), wsrc_c + (size_t)(cg - prm.cfull) * C::TAP_BYTES, C::TAP_BYTES, full);
            if (++ws == C::WS) { ws = 0; wph ^= 1; }
            continue;
          }
          for (int st = 0; st < kStagesPerChunk; ++st) {
            mbar_wait(smem_u32(&w_empty[ws]), wph ^ 1);
            const uint32_t full = smem_u32(&w_full[ws]);
            mbar_expect_tx(full, C::WST_BYTES);
            bulk_g2s(smem_u32(wst + ws * C::WST_BYTES), wsrc + (size_t)(c * kStagesPerChunk + st) * C::WST_BYTES,
                     C::WST_BYTES, full);
            if (++ws == C::WS) { ws = 0; wph ^= 1; }
          }
        }
      }
    }
  } else if (warp == kLoaderWarps + 4) {
    // ============ MMA issuer: the whole warp runs the (warp-uniform) control flow so that descriptors stay
    // in uniform registers; one elected lane issues tcgen05.mma / tcgen05.commit ============
    const int mw = 0;                                   // which issuing warp: patches p = mw (mod kMmaWarps)
    const bool leader = elect_one();
    // instruction descriptor: D=f32, A=B=(bf16|tf32), K-major both, N, M=128
    const uint32_t fmt = C::OP == OP_F16 ? 0u : (C::OP == OP_BF16 ? 1u : 2u);   // kind::f16: 0 = f16, 1 = bf16
    const uint32_t idesc =
        (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(C::N >> 3) << 17) | ((128u >> 4) << 24);
    const uint32_t halo_addr = smem_u32(halo), wst_addr = smem_u32(wst);
    int hs = 0, hph = 0, ws = 0, wph = 0, it = 0;
    for (int tile = tile0; tile < tile1; ++tile, ++it) {
      const int as = it & 1, aph = (it >> 1) & 1;
      mbar_wait(smem_u32(&acc_empty[as]), aph ^ 1);
      tc_fence_after();
      const uint32_t dbase = tmem_base + as * C::ACC_COLS;
      for (int c = 0; c < nchunks; ++c) {
        mbar_wait(smem_u32(&halo_full[hs]), hph);
        tc_fence_after();
        const uint64_t adesc0 = make_desc(halo_addr + hs * C::HALO_BYTES, C::HW * 16, C::RP * 16);
        if (C::KS == 3 && c_begin + c >= prm.cfull) {
          // centre-tap chunk: one N-wide MMA per output patch, A at the tap (1, 1, 1) of the halo
          mbar_wait(smem_u32(&w_full[ws]), wph);
          tc_fence_after();
          const uint64_t bdesc = make_desc(wst_addr + ws * C::WST_BYTES, C::N * 16, 128);
          if (leader) {
#pragma unroll
            for (int p = 0; p < C::P; ++p) {
              const int pd = p / C::NW, pw = p % C::NW;
              const uint32_t aoff = (uint32_t)(((pd + 1) * C::HH + 1) * C::RP + pw * 8 + 1);
              const uint32_t dcol = dbase + (uint32_t)((C::FOLD ? C::acc_block(pd, pw) : p) * C::N);
              const uint32_t acc_c = c > 0 ? 1u : 0u;      // (a split-K range may start inside the centre segment)
              if (C::BF16) tc_mma_f16(dcol, adesc0 + aoff, bdesc, idesc, acc_c);
              else tc_mma_tf32(dcol, adesc0 + aoff, bdesc, idesc, acc_c);
            }
            tc_commit(smem_u32(&w_empty[ws]));
          }
          __syncwarp();
          if (++ws == C::WS) { ws = 0; wph ^= 1; }
          if (leader) tc_commit(smem_u32(&halo_empty[hs]));
          __syncwarp();
          if (++hs == C::HS) { hs = 0; hph ^= 1; }
          continue;
        }
#pragma unroll
        for (int st = 0; st < C::TAPS / C::TPS; ++st) {
          mbar_wait(smem_u32(&w_full[ws]), wph);
          tc_fence_after();
          const uint64_t bdesc0 = make_desc(wst_addr + ws * C::WST_BYTES, C::NB * 16, 128);
          if (leader) {
            if constexpr (C::FOLD) {
              // stage st = kernel row kh; per (kh, kw) one B tile of 3N rows [kd=2 | kd=1 | kd=0]
              const int kh = st;
              constexpr uint32_t idesc_hi = (1u << 4) | ((128u >> 4) << 24);
              constexpr int kFoldG0 = (C::HD + 2) / 3, kFoldG1 = (C::HD + 1) / 3;      // slices = 0, 1 (mod 3)
              const uint32_t idf = idesc_hi | (fmt << 7) | (fmt << 10);
              const uint32_t id3 = idf | ((uint32_t)(3 * C::N >> 3) << 17), id2 = idf | ((uint32_t)(2 * C::N >> 3) << 17);
#pragma unroll
              for (int kw = 0; kw < 3; ++kw) {
                const uint64_t bdesc = bdesc0 + (uint64_t)(kw * (3 * C::TAP_BYTES >> 4));
                const bool first = c == 0 && st == 0 && kw == 0;
                // issue order: an MMA writes the accumulator blocks zi .. zi+2, so slices zi, zi+1 overlap in two of
                // them and back-to-back issue would chain every MMA on the completion of the previous one; walking the
                // slices with stride 3 (0,3,6,.. 1,4,7,.. 2,5,8,..) makes consecutive MMAs touch disjoint blocks.  The
                // very first step of a tile keeps the natural order: it also INITIALISES block zi+2 (accumulate = 0)
                // before slices zi+1, zi+2 add to it.
#pragma unroll
                for (int zj = 0; zj < C::HD; ++zj) {
                  const int zi = first ? zj : (zj < kFoldG0 ? 3 * zj : (zj < kFoldG0 + kFoldG1 ? 3 * (zj - kFoldG0) + 1
                                                                                              : 3 * (zj - kFoldG0 - kFoldG1) + 2));
#pragma unroll
                  for (int pw = 0; pw < C::NW; ++pw) {
                    const uint32_t aoff = (uint32_t)((zi * C::HH + kh) * C::RP + pw * 8 + kw);
                    const uint32_t dcol = dbase + (uint32_t)((pw * (C::TD + 4) + zi) * C::N);   // blocks of pd = zi-2..zi
                    if (!first) {
                      tc_mma_f16(dcol, adesc0 + aoff, bdesc, id3, 1u);
                    } else {
                      tc_mma_f16(dcol, adesc0 + aoff, bdesc, id2, 1u);                              // kd = 2, 1
                      tc_mma_f16(dcol + 2 * C::N, adesc0 + aoff, bdesc + (uint64_t)(2 * C::N), idesc, 0u);   // kd = 0
                    }
                  }
                }
              }
            } else {
#pragma unroll
            for (int tq = 0; tq < C::TPS; ++tq) {
              const int tap = st * C::TPS + tq;
              const int kd = tap / (C::KS * C::KS), kh = (tap / C::KS) % C::KS, kw = tap % C::KS;
              const uint64_t bdesc = bdesc0 + (uint64_t)(tq * (C::TAP_BYTES >> 4));
              const uint32_t acc = (c > 0 || tap > 0) ? 1u : 0u;
#pragma unroll
              for (int p = 0; p < C::P; ++p) {
                if ((p % kMmaWarps) != mw) continue;
                const int pd = p / C::NW, pw = p % C::NW;
                const uint32_t aoff = (uint32_t)(((pd + kd) * C::HH + kh) * C::RP + pw * 8 + kw);
                if (C::BF16) tc_mma_f16(dbase + p * C::N, adesc0 + aoff, bdesc, idesc, acc);
                else tc_mma_tf32(dbase + p * C::N, adesc0 + aoff, bdesc, idesc, acc);
              }
            }
            }
            tc_commit(smem_u32(&w_empty[ws]));
          }
          __syncwarp();
          if (++ws == C::WS) { ws = 0; wph ^= 1; }
        }
        if (leader) tc_commit(smem_u32(&halo_empty[hs]));
        __syncwarp();
        if (++hs == C::HS) { hs = 0; hph ^= 1; }
      }
      if (leader) tc_commit(smem_u32(&acc_full[as]));
      __syncwarp();
    }
  } else if (warp < 4 + kLoaderWarps) {
    // ============ epilogue (TMEM -> registers -> NDHWC global) ============
    // thread-loader form: warps 0-3, one per TMEM lane quarter; TMA form: warps 0-11, three per quarter, each taking
    // every third patch of a tile
    const int q = warp & 3;                 // TMEM lane quarter == warp % 4
    const int eg = warp >> 2, neg = prm.tma ? 1 + kLoaderWarps / 4 : 1;
    const bool wide_st = prm.act == 0 && prm.ksplit <= 1 && (prm.yp & 7) == 0 &&
                         (reinterpret_cast<uintptr_t>(prm.y) & 31) == 0;
    const int row = q * 32 + lane;          // patch row: h = row/8, w = row%8
    const int ph = row >> 3, pwv = row & 7;
    const long long S = (long long)prm.D * prm.H * prm.W * (prm.d2s ? 8 : 1);   // voxels of y per sample
    // global-average-pool partial sums: kept in registers across the tiles of one sample when N <= 64
    constexpr bool kGapPersist = C::N <= 32;      // (N = 64 would hold 64 accumulator registers and spill)
    constexpr int NJ = C::N / 16;
    float gsum[kGapPersist ? NJ : 1][16];
#pragma unroll
    for (int j = 0; j < (kGapPersist ? NJ : 1); ++j)
#pragma unroll
      for (int i = 0; i < 16; ++i) gsum[j][i] = 0.f;
    int gap_b = -1;
    auto flush_gap = [&](int bb) {
      if (prm.gap == nullptr || bb < 0) return;
#pragma unroll
      for (int j = 0; j < (kGapPersist ? NJ : 1); ++j)
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float a = warp_sum(gsum[j][i]);
          if (lane == 0 && nsp * C::N + j * 16 + i < prm.cout_real)
            atomicAdd(&prm.gap[(long long)bb * prm.cout_real + nsp * C::N + j * 16 + i], a);
          gsum[j][i] = 0.f;
        }
    };
    int it = 0;
    // running GroupNorm sums of this warp: kept ACROSS tiles and flushed when the chunk changes (a persistent CTA's
    // consecutive tiles usually lie in the same chunk) — the fp64 atomics all land on 2 * groups addresses
    int cur_chunk = -1;
    float s0 = 0.f, s1 = 0.f;
    for (int tile = tile0; tile < tile1; ++tile, ++it) {
      const int as = it & 1, aph = (it >> 1) & 1;
      int t = tile;
      const int wt = t % prm.ntw; t /= prm.ntw;
      const int ht = t % prm.nth; t /= prm.nth;
      const int dt = t % prm.ntd; t /= prm.ntd;
      const int b = t;
      if (kGapPersist && b != gap_b) { flush_gap(gap_b); gap_b = b; }
      mbar_wait(smem_u32(&acc_full[as]), aph);
      tc_fence_after();
#pragma unroll
      for (int j = 0; j < NJ; ++j) {
        // output column block -> (parity, channel offset) when the result is stored depth-to-space
        int ycol = nsp * C::N + j * 16, ep_d = 0, ep_h = 0, ep_w = 0;
        if (prm.d2s) {
          const int par = ycol / prm.Csub;
          ycol -= par * prm.Csub;
          ep_d = par >> 2; ep_h = (par >> 1) & 1; ep_w = par & 1;
        }
        const int ncol = min(16, prm.cout_real - (nsp * C::N + j * 16));    // real output channels in this block
        if (ncol <= 0) continue;
        float* ybase = prm.y;
        long long ypitch = prm.yp;
        if (prm.nyd > 1) {                  // which output piece this 16-column block belongs to
          int si = 0;
          while (si + 1 < prm.nyd && ycol >= prm.yde[si]) ++si;
          const int c0 = si > 0 ? prm.yde[si - 1] : 0;
          ybase = prm.yd[si]; ypitch = prm.yde[si] - c0; ycol -= c0;
        }
        float bv[16];
#pragma unroll
        for (int i = 0; i < 16; ++i) bv[i] = (prm.bias != nullptr && i < ncol) ? __ldg(prm.bias + ycol + i) : 0.f;
        float (&gs)[16] = gsum[kGapPersist ? j : 0];
#pragma unroll 1
        for (int p = eg; p < C::P; p += neg) {
          const int pd = p / C::NW, pw = p % C::NW;
          const int d = dt * C::TD + pd, h = ht * C::TH + ph, w = wt * C::TW + pw * 8 + pwv;
          const bool valid = d < prm.D && h < prm.H && w < prm.W;
          const long long vox =
              prm.d2s ? ((long long)(2 * d + ep_d) * (2 * prm.H) + (2 * h + ep_h)) * (2 * prm.W) + (2 * w + ep_w)
                      : ((long long)d * prm.H + h) * prm.W + w;
          float* yp = ybase + ((long long)b * S + vox) * ypitch + ycol;
          if (prm.stats != nullptr) {
            // the GroupNorm chunk of this patch's voxels; when any lane moves on to another chunk the whole warp
            // flushes its running sums (warp-reduced: two fp64 atomics per warp, not per lane)
            const int chunk = valid ? b * prm.groups + (int)((vox + prm.voff) / prm.vpc) : cur_chunk;
            if (__any_sync(0xffffffffu, chunk != cur_chunk && cur_chunk >= 0)) {
              flush_stats(prm.stats, cur_chunk, s0, s1, lane);
              cur_chunk = -1; s0 = 0.f; s1 = 0.f;
            }
            if (valid) cur_chunk = chunk;
          }
          float v[16];
          tc_ld16(tmem_base + ((uint32_t)(q * 32) << 16) + as * C::ACC_COLS + (C::FOLD ? C::acc_block(pd, pw) : p) * C::N + j * 16, v);
          if (valid && prm.ksplit > 1) {
            // partial sums of this K range -> workspace slice blockIdx.z
            float* dst = yp + (long long)blockIdx.z * prm.ws_slice;       // workspace slices are 128-byte aligned
            st256(dst, v[0], v[1], v[2], v[3], v[4], v[5], v[6], v[7]);
            st256(dst + 8, v[8], v[9], v[10], v[11], v[12], v[13], v[14], v[15]);
          } else if (valid && ncol < 16) {
            // narrow output (Cout < 16: the 2-3 channel output convs): scalar stores, optional sigmoid
#pragma unroll
            for (int i = 0; i < 16; ++i)
              if (i < ncol) {
                float o = v[i] + bv[i];
                if (prm.act == 1) o = 1.f / (1.f + expf(-o));
                if (prm.accumulate) o += yp[i];
                yp[i] = o;
                s0 += o;
                s1 += o * o;
                gs[i] += o;
              }
          } else if (valid && wide_st) {
            // plain epilogue (every conv of the training step but the sigmoid / accumulate forms): 2 x 256-bit stores
            float o[16];
            if (prm.accumulate) {
              // y += result (the second of two data gradients w.r.t. one tensor): the 64 bytes are fetched with four
              // 128-bit loads issued together
              float4 e[4];
#pragma unroll
              for (int i = 0; i < 4; ++i) e[i] = __ldcg(reinterpret_cast<const float4*>(yp) + i);
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                v[4 * i] += e[i].x; v[4 * i + 1] += e[i].y; v[4 * i + 2] += e[i].z; v[4 * i + 3] += e[i].w;
              }
            }
#pragma unroll
            for (int i = 0; i < 16; ++i) {
              o[i] = v[i] + bv[i];
              s0 += o[i];
              s1 += o[i] * o[i];
              gs[i] += o[i];
            }
            st256(yp, o[0], o[1], o[2], o[3], o[4], o[5], o[6], o[7]);
            st256(yp + 8, o[8], o[9], o[10], o[11], o[12], o[13], o[14], o[15]);
          } else if (valid) {
            float4* dst = reinterpret_cast<float4*>(yp);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              float4 o = make_float4(v[4 * i] + bv[4 * i], v[4 * i + 1] + bv[4 * i + 1], v[4 * i + 2] + bv[4 * i + 2],
                                     v[4 * i + 3] + bv[4 * i + 3]);
              if (prm.act == 1) {
                o.x = 1.f / (1.f + expf(-o.x)); o.y = 1.f / (1.f + expf(-o.y));
                o.z = 1.f / (1.f + expf(-o.z)); o.w = 1.f / (1.f + expf(-o.w));
              }
              if (prm.accumulate) {
                const float4 e = dst[i];
                o.x += e.x; o.y += e.y; o.z += e.z; o.w += e.w;
              }
              dst[i] = o;
              s0 += (o.x + o.y) + (o.z + o.w);
              s1 += (o.x * o.x + o.y * o.y) + (o.z * o.z + o.w * o.w);
              gs[4 * i] += o.x; gs[4 * i + 1] += o.y; gs[4 * i + 2] += o.z; gs[4 * i + 3] += o.w;
            }
          }
        }
        if (!kGapPersist && prm.gap != nullptr) {
          // wide layers: column sums flushed per tile (a tile lies in one sample) — into the CTA's shared-memory sums
          // when there is one sample (N = 64; written out once at the end), else straight to global memory
          const bool to_smem = C::N <= 64 && prm.B == 1;
          int i = 0;
          const float a = warp_colsum16(gs, lane, i);        // this lane's column of the 16 (lanes 2k, 2k+1: the same)
          if ((lane & 1) == 0 && nsp * C::N + j * 16 + i < prm.cout_real) {
            if (to_smem) atomicAdd(&cta_gap[j * 16 + i], a);
            else atomicAdd(&prm.gap[(long long)b * prm.cout_real + nsp * C::N + j * 16 + i], a);
          }
#pragma unroll
          for (int q2 = 0; q2 < 16; ++q2) gs[q2] = 0.f;
          if (to_smem && lane == 0) *cta_gap_b = b;
        }
      }
      // release the accumulator stage as soon as TMEM has been read
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(smem_u32(&acc_empty[as]));
    }
    if (prm.stats != nullptr) flush_stats_cta(prm.stats, cur_chunk, s0, s1, lane, cta_stat, cta_stat_tag);
    if (kGapPersist && prm.gap != nullptr && gap_b >= 0) {
      // all epilogue warps end on the same tile, hence the same sample
#pragma unroll
      for (int j = 0; j < NJ; ++j)
#pragma unroll
        for (int i = 0; i < 16; ++i) {
          const float a = warp_sum(gsum[j][i]);
          if (lane == 0) atomicAdd(&cta_gap[j * 16 + i], a);
        }
      if (lane == 0) *cta_gap_b = gap_b;
    }
  }

  // ---- teardown
  tc_fence_before();
  __syncthreads();
  if (threadIdx.x < 4 && prm.stats != nullptr && cta_stat_tag[threadIdx.x] >= 0) {
    atomicAdd(&prm.stats[2 * cta_stat_tag[threadIdx.x]], cta_stat[2 * threadIdx.x]);
    atomicAdd(&prm.stats[2 * cta_stat_tag[threadIdx.x] + 1], cta_stat[2 * threadIdx.x + 1]);
  }
  if (C::N <= 64 && threadIdx.x >= 32 && threadIdx.x < 32 + C::N && prm.gap != nullptr && *cta_gap_b >= 0) {
    const int i = threadIdx.x - 32;
    if (nsp * C::N + i < prm.cout_real)
      atomicAdd(&prm.gap[(long long)*cta_gap_b * prm.cout_real + nsp * C::N + i], cta_gap[i]);
  }
  if (warp == kLoaderWarps + 5) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512));
  }
}

// ------------------------------------------------------------------------------------------ split-K epilogue
// y = sum of the split-K workspace slices + bias, with the GroupNorm chunk statistics and per-channel sums of y.
// grid = (B * G, segments): blockIdx.x = contiguous chunk of a sample (G = groups, or 8 pseudo-chunks), blockIdx.y
// = 8192-element segment of it; statistics / GAP are accumulated with atomics into buffers zeroed by the caller.
__global__ void __launch_bounds__(256)
    conv_finish_kernel(float* __restrict__ y, const float* __restrict__ ws, int ksplit, long long ws_slice,
                       const float* __restrict__ bias, double* __restrict__ stats, float* __restrict__ gap,
                       long long L, int C, int G, long long shift, long long n_local, int chunk0) {
  pdl_trigger();
  pdl_wait();
  extern __shared__ float sgap[];                  // [C]
  __shared__ double red[64];
  const int chunk = blockIdx.x + chunk0;           // slab form: the grid starts at the first intersecting chunk
  const int b = chunk / G, g = chunk % G;
  // depth-slab form (n_local >= 0, batch 1): y holds the elements [shift, shift + n_local) of the volume whose chunks
  // (G, L) describe; a CTA covers the part of its chunk's segment that lies inside
  long long e_lo = 0, e_hi = L, sh = 0;
  if (n_local >= 0) {
    sh = shift;
    e_lo = max(0LL, shift - (long long)g * L);
    e_hi = min(L, shift + n_local - (long long)g * L);
  }
  const long long seg0 = e_lo + (long long)blockIdx.y * 8192, seg1 = min(e_hi, seg0 + 8192);
  if (seg0 >= seg1) return;                        // CTA-uniform
  for (int i = threadIdx.x; i < C; i += 256) sgap[i] = 0.f;
  __syncthreads();
  const long long off = ((long long)b * G + g) * L - sh;
  float* yc = y + off;
  const long long e0 = (long long)g * L;           // element offset inside the sample (channel = (e0 + e) % C)
  double d[2] = {0.0, 0.0};
  for (long long e = seg0 + threadIdx.x * 4LL; e < seg1; e += 256 * 4) {
    // all slices' loads are issued before the first add (ksplit <= 8): one L2 round trip per element, not ksplit
    float4 t[8];
#pragma unroll
    for (int z = 0; z < 8; ++z)
      if (z < ksplit) t[z] = ld_stream(reinterpret_cast<const float4*>(ws + (long long)z * ws_slice + off + e));
    float4 v = t[0];
#pragma unroll
    for (int z = 1; z < 8; ++z)
      if (z < ksplit) { v.x += t[z].x; v.y += t[z].y; v.z += t[z].z; v.w += t[z].w; }
    const int c = (int)((e0 + e) % C);
    if (bias != nullptr) { v.x += bias[c]; v.y += bias[c + 1]; v.z += bias[c + 2]; v.w += bias[c + 3]; }
    *reinterpret_cast<float4*>(yc + e) = v;
    d[0] += (double)((v.x + v.y) + (v.z + v.w));
    d[1] += (double)((v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w));
    if (gap != nullptr) {
      atomicAdd(&sgap[c], v.x); atomicAdd(&sgap[c + 1], v.y); atomicAdd(&sgap[c + 2], v.z); atomicAdd(&sgap[c + 3], v.w);
    }
  }
  block_sum<2, double>(d, red);
  if (stats != nullptr && threadIdx.x == 0) {      // G == groups when statistics are requested
    atomicAdd(&stats[2 * chunk], d[0]);
    atomicAdd(&stats[2 * chunk + 1], d[1]);
  }
  __syncthreads();
  if (gap != nullptr)
    for (int i = threadIdx.x; i < C; i += 256) atomicAdd(&gap[(long long)b * C + i], sgap[i]);
}

// ------------------------------------------------------------------------------------------ packing
// wp[ns][c][tap][pl][n][j] = op( w[tw(tap)*wtap + (CK*c + T*pl + j)*sw_in + (ns*N+n)*sw_out] ),  op = bf16 | tf32
__device__ __forceinline__ float pack_s1_elem(const float* __restrict__ w, long long i, int T, int taps, int Cin, int N,
                                              long long wtap, int sw_in, int sw_out, int flip, int cin_real,
                                              int cout_real) {
  const int nch = Cin / (2 * T);
  long long r = i;
  const int j = (int)(r % T); r /= T;
  const int n = (int)(r % N); r /= N;
  const int pl = (int)(r % 2); r /= 2;
  int tap = (int)(r % taps); r /= taps;
  const int c = (int)(r % nch); r /= nch;
  const int ns = (int)r;
  if (flip) tap = taps - 1 - tap;
  const int ci = 2 * T * c + T * pl + j, co = ns * N + n;
  return (ci < cin_real && co < cout_real)
             ? w[(long long)tap * wtap + (long long)ci * sw_in + (long long)co * sw_out] : 0.f;
}

// kd-folded layout (TcCfg::FOLD): wp[ns][c][kh*3+kw][pl][(2-kd)*N + n][j] — per (kh, kw) one B tile of 3N rows
__device__ __forceinline__ float pack_s1_fold_elem(const float* __restrict__ w, long long i, int T, int Cin, int N,
                                                   long long wtap, int sw_in, int sw_out, int flip, int cin_real,
                                                   int cout_real) {
  const int nch = Cin / (2 * T);
  long long r = i;
  const int j = (int)(r % T); r /= T;
  const int nn = (int)(r % (3 * N)); r /= 3 * N;
  const int pl = (int)(r % 2); r /= 2;
  const int khw = (int)(r % 9); r /= 9;
  const int c = (int)(r % nch); r /= nch;
  const int ns = (int)r;
  const int kd = 2 - nn / N, n = nn % N;
  int tap = kd * 9 + khw;
  if (flip) tap = 26 - tap;
  const int ci = 2 * T * c + T * pl + j, co = ns * N + n;
  return (ci < cin_real && co < cout_real)
             ? w[(long long)tap * wtap + (long long)ci * sw_in + (long long)co * sw_out] : 0.f;
}

template <int OP>
__device__ __forceinline__ void pack_store(void* __restrict__ wp, long long i, float v) {
  if (OP == OP_BF16) {
    reinterpret_cast<__nv_bfloat16*>(wp)[i] = __float2bfloat16_rn(v);
  } else if (OP == OP_F16) {
    reinterpret_cast<__half*>(wp)[i] = __float2half_rn(v);
  } else {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(v));
    reinterpret_cast<float*>(wp)[i] = __uint_as_float(u);
  }
}

template <int OP>
__global__ void tc_pack_kernel(const float* __restrict__ w, void* __restrict__ wp, int taps, int Cin, int Cout, int N,
                               long long wtap, int sw_in, int sw_out, int flip, int cin_real, int cout_real,
                               int fold) {
  constexpr int T = OP != OP_TF32 ? 8 : 4;
  const long long total = (long long)taps * Cin * Cout;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x)
    pack_store<OP>(wp, i, fold ? pack_s1_fold_elem(w, i, T, Cin, N, wtap, sw_in, sw_out, flip, cin_real, cout_real)
                               : pack_s1_elem(w, i, T, taps, Cin, N, wtap, sw_in, sw_out, flip, cin_real, cout_real));
}

// every layer's operand re-layout in ONE launch (after the optimiser step): block -> job by binary search over the
// jobs' first-block table, kPackPerBlock elements per block
constexpr int kPackPerBlock = 2048;
__global__ void __launch_bounds__(256) pack_many_kernel(const PackJob* __restrict__ jobs, int njobs) {
  int lo = 0, hi = njobs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].block0 <= (long long)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const PackJob jb = jobs[lo];
  const long long base = ((long long)blockIdx.x - jb.block0) * kPackPerBlock;
  const int T = jb.op != OP_TF32 ? 8 : 4;
  for (int e = threadIdx.x; e < kPackPerBlock; e += 256) {
    const long long i = base + e;
    if (i >= jb.total) break;
    const float v =
        jb.s2 == 1 ? pack_s2_elem(jb.w, i, T, jb.up, jb.Cin, jb.Cout, jb.N, jb.wtap, jb.sw_in, jb.sw_out, jb.aux)
        : jb.s2 == 2 ? pack_s1_fold_elem(jb.w, i, T, jb.Cin, jb.N, jb.wtap, jb.sw_in, jb.sw_out, jb.aux, jb.cin_real,
                                         jb.cout_real)
                     : pack_s1_elem(jb.w, i, T, jb.taps, jb.Cin, jb.N, jb.wtap, jb.sw_in, jb.sw_out, jb.aux,
                                    jb.cin_real, jb.cout_real);
    if (jb.op == OP_BF16) pack_store<OP_BF16>(jb.wp, i, v);
    else if (jb.op == OP_F16) pack_store<OP_F16>(jb.wp, i, v);
    else pack_store<OP_TF32>(jb.wp, i, v);
  }
}

// ------------------------------------------------------------------------------------------ host
// operand type of the conv MMAs, per pass: forward defaults to tf32 (north_star's 2e-3 per-layer tolerance,
// argmax agreement), the data gradient to bf16 (1e-2); fp32 accumulation in TMEM either way
static int g_fwd_op = OP_F16, g_bwd_op = OP_BF16;

EncodeTiledFn tma_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (fn == nullptr) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)p;
  }
  return fn;
}

static int pick_n(int Cout) {      // widest N tile that divides the (16-padded) output channels
  if (Cout % 128 == 0) return 128;
  if (Cout % 64 == 0) return 64;
  if (Cout % 32 == 0) return 32;
  return 16;
}

// 16-bit operands need whole 16-channel K steps: Cin % 16 == 0, or a narrow input (Cin < 8) zero-padded to 16
static int operand_type(const ConvGeom& g) {
  const int op = g.bwd ? g_bwd_op : g_fwd_op;
  return (op != OP_TF32 && (g.Cin % 16 == 0 || (g.mode == CONV_S1 && g.Cin < 8))) ? op : OP_TF32;
}
static int pad_cin(const ConvGeom& g) {
  const int ck = operand_type(g) == OP_TF32 ? 8 : 16;
  return (g.Cin + ck - 1) / ck * ck;
}
static int pad_cout(int c) { return (c + 15) / 16 * 16; }

// kd-folded variant of the 3x3x3 kernel (TcCfg::FOLD): narrow output tiles with 16-bit operands.  On by default
// (b3d_set_conv_kdfold switches it); the packed weight layout depends on it.
static int g_kdfold = 1;
static bool use_fold(const ConvGeom& g) {
  if (!g_kdfold || g.mode != CONV_S1 || g.k != 3 || operand_type(g) == OP_TF32) return false;
  const int n = pick_n(pad_cout(g.Cout));
  return n == 16 || n == 32;
}

// virtual (stride-1) problem of a conv geometry: S1 as is; DOWN / UP = 2x2x2 conv on the coarse grid (conv_s2.cu)
struct TcProblem {
  int ks, hb, Cin, Cout, D, H, W, s2d, d2s, Csub;
};
static TcProblem tc_problem(const ConvGeom& g) {
  TcProblem q;
  memset(&q, 0, sizeof(q));
  if (g.mode == CONV_S1) {
    q.ks = g.k; q.hb = g.k == 2 ? g.pad : g.k / 2; q.Cin = pad_cin(g); q.Cout = pad_cout(g.Cout);
    q.D = g.Do; q.H = g.Ho; q.W = g.Wo;
  } else if (g.mode == CONV_DOWN) {
    q.ks = 2; q.hb = 0; q.Cin = 8 * g.Cin; q.Cout = pad_cout(g.Cout); q.D = g.Do; q.H = g.Ho; q.W = g.Wo;
    q.s2d = 1; q.Csub = g.Cin;
  } else {
    q.ks = 2; q.hb = 1; q.Cin = g.Cin; q.Cout = 8 * g.Cout; q.D = g.Do / 2; q.H = g.Ho / 2; q.W = g.Wo / 2;
    q.d2s = 1; q.Csub = g.Cout;
  }
  return q;
}

// g.bwd marks the backward pass (precision choice); chunks of CK channels must not straddle a parity block
bool tc_conv_supported(const ConvGeom& g) {
  if (g.mode == CONV_S1)     // narrow inputs (Cin < 8) / outputs (Cout < 16) run zero-padded to one K step / N tile
    return (g.k == 3 || g.k == 1) && g.Cin >= 1 && g.Cout >= 1 && (g.Cin % 8 == 0 || g.Cin < 8) &&
           (g.Cout % 16 == 0 || g.Cout < 16);
  // stride-2 family.  (Narrow outputs only occur in the VAE bottleneck, 16^3 -> 8^3 x 8 and 16^3 x 128 -> 8^3 x 1:
  // a few hundred output voxels with a long reduction — those run on conv_gather_splitk_kernel instead.)
  return g.k == 3 && g.Cin % 8 == 0 && g.Cin >= 8 && g.Cout % 16 == 0 && g.Cout >= 16;
}

size_t tc_packed_weight_elems(const ConvGeom& g) {
  if (g.mode != CONV_S1) return (size_t)64 * pad_cout(g.Cin) * pad_cout(g.Cout);   // symmetric in the channel roles
  return (size_t)g.k * g.k * g.k * ((g.Cin + 15) / 16 * 16) * pad_cout(g.Cout);   // room for either operand type
}

// the re-layout of one layer as a PackJob (block0 is filled in by the caller); the single place that knows the
// parameters of both pack kernels
int tc_pack_job(const ConvGeom& g, const float* w, float* wp, PackJob* jb) {
  B3D_REQUIRE(tc_conv_supported(g), B3D_ERR_UNSUPPORTED, "pack_weights: shape not on the tcgen05 path");
  memset(jb, 0, sizeof(*jb));
  jb->w = w; jb->wp = wp; jb->op = operand_type(g);
  jb->wtap = g.wtap; jb->sw_in = g.sw_in; jb->sw_out = g.sw_out;
  if (g.mode != CONV_S1) {
    const int up = g.mode == CONV_UP ? 1 : 0;
    const int ntd = (g.Cout + 15) / 16 * 16;
    const int K = up ? g.Cin : 8 * g.Cin, NT = up ? 8 * g.Cout : ntd;
    jb->s2 = 1; jb->up = up; jb->Cin = g.Cin; jb->Cout = g.Cout; jb->N = tc_pick_n(NT); jb->aux = ntd;
    jb->total = 8LL * K * NT;
  } else {
    jb->taps = g.k * g.k * g.k; jb->Cin = pad_cin(g); jb->Cout = pad_cout(g.Cout); jb->N = pick_n(jb->Cout);
    jb->aux = g.flip; jb->cin_real = g.Cin; jb->cout_real = g.Cout;
    jb->total = (long long)jb->taps * jb->Cin * jb->Cout;
    if (use_fold(g)) jb->s2 = 2;
  }
  return B3D_OK;
}
long long tc_pack_job_blocks(const PackJob& jb) { return (jb.total + kPackPerBlock - 1) / kPackPerBlock; }

int launch_tc_pack_many(const PackJob* jobs_dev, int njobs, long long blocks, cudaStream_t s) {
  if (njobs <= 0 || blocks <= 0) return B3D_OK;
  pack_many_kernel<<<(unsigned)blocks, 256, 0, s>>>(jobs_dev, njobs);
  B3D_LAUNCH_CHECK("pack_many");
  return B3D_OK;
}

int launch_tc_pack_weights(const ConvGeom& g, const float* w, float* wp, cudaStream_t s) {
  B3D_REQUIRE(tc_conv_supported(g), B3D_ERR_UNSUPPORTED, "pack_weights: shape not on the tcgen05 path");
  const int op = operand_type(g);
  if (g.mode != CONV_S1) return launch_pack_s2(g, w, wp, op, s);
  const int taps = g.k * g.k * g.k, cin = pad_cin(g), cout = pad_cout(g.Cout);
  const long long total = (long long)taps * cin * cout;
  const unsigned grid = (unsigned)((total + 255) / 256 < 4096 ? (total + 255) / 256 : 4096);
#define B3D_PACK(OPV)                                                                                          \
  tc_pack_kernel<OPV><<<grid, 256, 0, s>>>(w, wp, taps, cin, cout, pick_n(cout), g.wtap, g.sw_in, g.sw_out, g.flip, \
                                           g.Cin, g.Cout, use_fold(g) ? 1 : 0)
  if (op == OP_BF16) B3D_PACK(OP_BF16);
  else if (op == OP_F16) B3D_PACK(OP_F16);
  else B3D_PACK(OP_TF32);
#undef B3D_PACK
  B3D_LAUNCH_CHECK("tc_pack");
  return B3D_OK;
}

// split-K workspace: 64 MB per device, allocated lazily (never while the stream is being captured)
constexpr long long kSplitWsElems = 16LL << 20;
static float* splitk_workspace(cudaStream_t s) {
  static float* ws[16] = {nullptr};
  int dev = 0;
  cudaGetDevice(&dev);
  if (dev < 0 || dev >= 16) return nullptr;
  if (ws[dev] == nullptr) {
    cudaStreamCaptureStatus st = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(s, &st) != cudaSuccess || st != cudaStreamCaptureStatusNone) return nullptr;
    if (cudaMalloc(&ws[dev], sizeof(float) * kSplitWsElems) != cudaSuccess) { cudaGetLastError(); ws[dev] = nullptr; }
  }
  return ws[dev];
}

// tensor map of a P16 operand [B, D, H, C/8, W, 8] for boxes of bw voxels x `planes` x bh x bd: the innermost dimension
// is the (w, 8 channels) run of a plane row counted in 32-bit words (4 per 16-byte cell; a box extent is limited to 256
// ELEMENTS, so words instead of halves allow rows of up to 64 voxels) -> dims (4W, C/8, H, D, B), coordinate 4*w.
int make_p16_map(CUtensorMap* tm, const void* base, int bf16, int B, int D, int H, int W, int C8, int bw, int planes,
                 int bh, int bd) {
  (void)bf16;
  EncodeTiledFn enc = tma_encode_fn();
  B3D_REQUIRE(enc != nullptr, B3D_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  B3D_REQUIRE(4 * bw <= 256 && planes <= 256 && bh <= 256 && bd <= 256, B3D_ERR_UNSUPPORTED, "P16 map: box too large");
  const cuuint64_t row = (cuuint64_t)W * 16;
  const cuuint64_t dims[5] = {(cuuint64_t)W * 4, (cuuint64_t)C8, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)B};
  const cuuint64_t strides[4] = {row, row * C8, row * C8 * H, row * C8 * H * D};
  const cuuint32_t box[5] = {(cuuint32_t)(4 * bw), (cuuint32_t)planes, (cuuint32_t)bh, (cuuint32_t)bd, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, (void*)base,
                         dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B3D_REQUIRE(r == CUDA_SUCCESS, B3D_ERR_CUDA, "cuTensorMapEncodeTiled(P16) failed (%d)", (int)r);
  return B3D_OK;
}

// the same tensor with the dimensions in another ORDER, so that one box lands in shared memory as [o3][o2][o1][w]:
// order = 0: (4W, H, C/8, D, B) -> a box {4bw, bh, planes, bd} is [d][plane][h][w] (x tile of the kd-in-M weight gradient);
// order = 1: (4W, H, D, C/8, B) -> a box {4bw, bh, bd, planes} is [plane][d][h][w] (its dy tile, all planes at once)
int make_p16_map_perm(CUtensorMap* tm, const void* base, int order, int B, int D, int H, int W, int C8, int bw, int planes,
                      int bh, int bd) {
  EncodeTiledFn enc = tma_encode_fn();
  B3D_REQUIRE(enc != nullptr, B3D_ERR_CUDA, "cuTensorMapEncodeTiled entry point not available");
  B3D_REQUIRE(4 * bw <= 256 && planes <= 256 && bh <= 256 && bd <= 256, B3D_ERR_UNSUPPORTED, "P16 map: box too large");
  const cuuint64_t row = (cuuint64_t)W * 16;
  const cuuint64_t sp = row, sh = row * C8, sd = row * C8 * H, sb = row * C8 * H * D;
  cuuint64_t dims[5] = {(cuuint64_t)W * 4, (cuuint64_t)H, 0, 0, (cuuint64_t)B};
  cuuint64_t strides[4] = {sh, 0, 0, sb};
  cuuint32_t box[5] = {(cuuint32_t)(4 * bw), (cuuint32_t)bh, 0, 0, 1};
  if (order == 0) {
    dims[2] = (cuuint64_t)C8; dims[3] = (cuuint64_t)D; strides[1] = sp; strides[2] = sd;
    box[2] = (cuuint32_t)planes; box[3] = (cuuint32_t)bd;
  } else {
    dims[2] = (cuuint64_t)D; dims[3] = (cuuint64_t)C8; strides[1] = sd; strides[2] = sp;
    box[2] = (cuuint32_t)bd; box[3] = (cuuint32_t)planes;
  }
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_UINT32, 5, (void*)base,
                         dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                         CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  B3D_REQUIRE(r == CUDA_SUCCESS, B3D_ERR_CUDA, "cuTensorMapEncodeTiled(P16, permuted) failed (%d)", (int)r);
  return B3D_OK;
}

template <class C>
static int launch_cfg(const ConvGeom& g, const TcProblem& q, const float* x, const float* wp, const float* bias,
                      float* y, double* stats, float* gap, cudaStream_t s, const TcSources* srcs) {
  TcParams p;
  memset(&p, 0, sizeof(p));
  TcMaps maps;
  memset(&maps, 0, sizeof(maps));
  if (srcs != nullptr) {
    if constexpr (!C::BF16) {
      set_error("tcgen05 conv: P16 operands need a 16-bit operand type");
      return B3D_ERR_UNSUPPORTED;
    } else {
      B3D_REQUIRE((C::OP == OP_BF16) == (srcs->bf16 != 0), B3D_ERR_DTYPE,
                  "tcgen05 conv: P16 operand type (%s) does not match the pass's MMA operand type",
                  srcs->bf16 ? "bf16" : "fp16");
      p.x16 = 1; p.nsrc = srcs->n; p.tma = q.s2d ? 0 : 1;
      int cum = 0;
      for (int i = 0; i < srcs->n; ++i) {
        B3D_REQUIRE(srcs->C[i] % 16 == 0, B3D_ERR_UNSUPPORTED, "tcgen05 conv: P16 sources need channels %% 16 == 0");
        cum += srcs->C[i];
        p.src[i] = srcs->p[i]; p.cend[i] = cum; p.sc8[i] = srcs->C[i] / 8;
        if (p.tma)
          B3D_TRY(make_p16_map(&maps.m[i], srcs->p[i], srcs->bf16, g.B, g.Di, g.Hi, g.Wi, srcs->C[i] / 8, C::HW, 2, C::HH,
                               C::HD));
      }
    }
  }
  p.x = x; p.wp = wp; p.bias = bias; p.y = y; p.stats = stats; p.gap = gap;
  p.B = g.B; p.D = q.D; p.H = q.H; p.W = q.W; p.Cin = q.Cin; p.Cout = q.Cout; p.xp = g.xp; p.yp = g.yp;
  p.ntd = (q.D + C::TD - 1) / C::TD; p.nth = (q.H + C::TH - 1) / C::TH; p.ntw = (q.W + C::TW - 1) / C::TW;
  p.ntiles = g.B * p.ntd * p.nth * p.ntw;
  p.accumulate = g.accumulate; p.groups = g.groups > 0 ? g.groups : 1;
  p.vpc = (g.stat_total > 0 ? g.stat_total : (long long)g.Do * g.Ho * g.Wo) / p.groups;
  p.voff = g.stat_total > 0 ? g.stat_off : 0;
  p.s2d = q.s2d; p.d2s = q.d2s; p.Csub = q.Csub;
  p.Din = g.Di; p.doff = g.doff;
  p.cfull = (q.Cin - (q.ks == 3 ? g.c_center : 0)) / C::CK;
  p.wpc = g.wp_center;
  p.nyd = g.nyd;
  for (int i = 0; i < g.nyd && i < 4; ++i) { p.yd[i] = g.yd[i]; p.yde[i] = g.yde[i]; }
  p.cin_real = g.mode == CONV_S1 ? g.Cin : q.Cin; p.cout_real = g.mode == CONV_UP ? q.Cout : g.Cout; p.act = g.act;
  static bool attr_set = false;
  if (!attr_set) {
    B3D_TRY(cuda_ok(cudaFuncSetAttribute(conv_tc_kernel<C>, cudaFuncAttributeMaxDynamicSharedMemorySize, C::SMEM),
                    "cudaFuncSetAttribute(conv_tc)"));
    attr_set = true;
  }
  const int nsplit = q.Cout / C::N;
  dim3 grid((unsigned)(p.ntiles < sm_count() ? p.ntiles : sm_count()), (unsigned)nsplit, 1);
  if (nsplit > 1) grid.x = (grid.x + nsplit - 1) / nsplit;   // keep ~one persistent CTA per SM in total
  // split-K: small volumes (the 16^3 level, thin inference slabs) give far fewer tiles than SMs while their
  // reductions are the longest of the net (Cin up to 512): spread the K chunks over blockIdx.z.  Partial results go
  // through a per-device workspace that is allocated on first use (outside CUDA-graph capture) and kept.
  const int nchunks = q.Cin / C::CK;
  const long long S = (long long)g.Do * g.Ho * g.Wo;
  const long long out_elems = (long long)g.B * S * g.Cout;
  p.ksplit = 1; p.kchunks = nchunks; p.ws_slice = 0;
  const int ctas = (int)(grid.x * grid.y);
  float* ws = nullptr;
  if (ctas * 2 <= sm_count() && nchunks >= 8 && g.act == 0 && !g.accumulate && g.Cout % 16 == 0 && g.yp == g.Cout &&
      g.nyd <= 1 &&
      (S * g.Cout) % 32 == 0 && (stats == nullptr || p.groups == 8 || S % p.groups == 0) &&
      (stats == nullptr || g.stat_total == 0 || (g.B == 1 && (g.stat_total * g.Cout) % (4LL * p.groups) == 0))) {
    int ks = sm_count() / ctas;
    if (ks > nchunks / 4) ks = nchunks / 4;
    if (ks > 8) ks = 8;
    while (ks >= 2 && ks * out_elems > kSplitWsElems) --ks;
    if (ks >= 2 && (ws = splitk_workspace(s)) != nullptr) {
      p.kchunks = (nchunks + ks - 1) / ks;
      p.ksplit = (nchunks + p.kchunks - 1) / p.kchunks;
    }
  }
  if (p.ksplit > 1) {
    grid.z = (unsigned)p.ksplit;
    p.bias = nullptr; p.stats = nullptr; p.gap = nullptr;
    p.y = ws; p.ws_slice = out_elems;
  }
  // programmatic dependent launch (common.cuh): the CTAs' prologue overlaps the tail of the previous kernel
  B3D_TRY(cuda_ok(launch_pdl(conv_tc_kernel<C>, grid, dim3(kTcThreads), C::SMEM, s, p, maps), "launch conv_tc"));
  B3D_LAUNCH_CHECK("conv_tc");
  if (p.ksplit > 1) {
    const int G = stats != nullptr ? (g.groups > 0 ? g.groups : 1) : 8;
    const bool slab = stats != nullptr && g.stat_total > 0;       // chunks of the whole volume, window of this slab
    const long long L = (slab ? g.stat_total : S) * g.Cout / G;
    const long long span = slab && out_elems < L ? out_elems : L;  // longest part of a chunk a CTA row can hold
    const long long sh = slab ? g.stat_off * g.Cout : 0;
    const int c0 = slab ? (int)(sh / L) : 0, nc = slab ? (int)((sh + out_elems - 1) / L) - c0 + 1 : g.B * G;
    launch_pdl(conv_finish_kernel, dim3(nc, (unsigned)((span + 8191) / 8192)), 256, sizeof(float) * g.Cout, s, y, ws, p.ksplit, out_elems, bias, stats, gap, L, g.Cout, G, sh, slab ? out_elems : -1, c0);
    B3D_LAUNCH_CHECK("conv_finish");
  }
  return B3D_OK;
}

template <int KS, int HB, int BF16>
static int dispatch_n(const ConvGeom& g, const TcProblem& q, const float* x, const float* wp, const float* bias,
                      float* y, double* stats, float* gap, cudaStream_t s, const TcSources* srcs) {
  const int n = pick_n(q.Cout);
  if constexpr (KS == 3 && HB == 1 && BF16 != OP_TF32) {
    if (use_fold(g)) {
      if (n == 16) return launch_cfg<TcCfg<16, 8, 1, KS, HB, BF16, 1>>(g, q, x, wp, bias, y, stats, gap, s, srcs);
      return launch_cfg<TcCfg<32, 4, 1, KS, HB, BF16, 1>>(g, q, x, wp, bias, y, stats, gap, s, srcs);
    }
  }
  if (n == 128) return launch_cfg<TcCfg<128, 2, 1, KS, HB, BF16>>(g, q, x, wp, bias, y, stats, gap, s, srcs);
  if constexpr (!(KS == 2 && HB == 1)) {   // the depth-to-space form always has N = 8*Cp = multiple of 128
    if (n == 64) return launch_cfg<TcCfg<64, 2, 2, KS, HB, BF16>>(g, q, x, wp, bias, y, stats, gap, s, srcs);
    if (n == 32) return launch_cfg<TcCfg<32, 4, 2, KS, HB, BF16>>(g, q, x, wp, bias, y, stats, gap, s, srcs);
    return launch_cfg<TcCfg<16, 4, 2, KS, HB, BF16>>(g, q, x, wp, bias, y, stats, gap, s, srcs);
  }
  set_error("tcgen05 conv: unexpected N tile");
  return B3D_ERR_UNSUPPORTED;
}

// conv on the tensor cores with pre-packed weights: stride-1 k in {1,3}; stride-2 family (mode DOWN / UP) as a
// 2x2x2 stride-1 conv over the coarse grid with space-to-depth input / depth-to-space output addressing
int launch_conv_tc(const ConvGeom& g, const float* x, const float* wp, const float* bias, float* y, double* stats,
                   float* gap, cudaStream_t s, const TcSources* srcs) {
  B3D_REQUIRE(tc_conv_supported(g), B3D_ERR_UNSUPPORTED, "conv: shape not supported by the tcgen05 path");
  B3D_REQUIRE(g.act == 0 || (g.act == 1 && g.mode == CONV_S1), B3D_ERR_UNSUPPORTED,
              "tcgen05 conv: only the sigmoid epilogue of stride-1 convs is built");
  B3D_REQUIRE(srcs != nullptr || g.Cin < 8 || (g.xp % 8 == 0 && ((uintptr_t)x & 31) == 0), B3D_ERR_LAYOUT,
              "tcgen05 conv: x must be 32-byte aligned with a channel pitch multiple of 8");
  B3D_REQUIRE(g.Cout < 16 || (g.yp % 4 == 0 && ((uintptr_t)y & 15) == 0), B3D_ERR_LAYOUT,
              "tcgen05 conv: y must be 16-byte aligned with a channel pitch multiple of 4");
  B3D_REQUIRE(((uintptr_t)wp & 15) == 0, B3D_ERR_LAYOUT, "tcgen05 conv: packed weights must be 16-byte aligned");
  const TcProblem q = tc_problem(g);
  B3D_REQUIRE(gap == nullptr || g.mode == CONV_S1, B3D_ERR_UNSUPPORTED, "tcgen05 conv: GAP only for stride 1");
  const int op = operand_type(g);
#define B3D_TC_DISPATCH(KS, HB)                                                                   \
  return op == OP_BF16 ? dispatch_n<KS, HB, OP_BF16>(g, q, x, wp, bias, y, stats, gap, s, srcs)          \
         : op == OP_F16 ? dispatch_n<KS, HB, OP_F16>(g, q, x, wp, bias, y, stats, gap, s, srcs)          \
                        : dispatch_n<KS, HB, OP_TF32>(g, q, x, wp, bias, y, stats, gap, s, srcs)
  if (q.ks == 3) { B3D_TC_DISPATCH(3, 1); }
  if (q.ks == 1) { B3D_TC_DISPATCH(1, 0); }
  if (q.hb == 1) { B3D_TC_DISPATCH(2, 1); }
  B3D_TC_DISPATCH(2, 0);
#undef B3D_TC_DISPATCH
}

int tc_operand_type(const ConvGeom& g) { return operand_type(g); }
int tc_pick_n(int Cout) { return pick_n(Cout); }

}  // namespace b3d

// operand type of the tcgen05 conv MMAs (0 = tf32, 1 = bf16, 2 = fp16), separately for the forward pass and for
// the data gradient; fp32 accumulation in TMEM either way.  fp16 has TF32's 11-bit significand at bf16's cost
// (half the shared-memory bytes per MAC) and is used for the FORWARD operands, whose range is bounded by
// GroupNorm; gradients keep bf16's exponent range.
extern "C" int b3d_set_conv_precision(int fwd, int bwd) {
  if (fwd < 0 || fwd > 2 || bwd < 0 || bwd > 2) { b3d::set_error("conv precision: 0 tf32, 1 bf16, 2 fp16"); return B3D_ERR_ARG; }
  b3d::g_fwd_op = fwd;
  b3d::g_bwd_op = bwd;
  return 0;
}
extern "C" int b3d_get_conv_precision(void) { return b3d::g_fwd_op | (b3d::g_bwd_op << 4); }

// kd-folded 3x3x3 kernel for output tiles of 16 / 32 channels (see the header comment of this file).  Changes the
// packed weight layout of those layers: re-pack after switching.  Returns the previous setting.
extern "C" int b3d_set_conv_kdfold(int on) {
  const int prev = b3d::g_kdfold;
  b3d::g_kdfold = on ? 1 : 0;
  return prev;
}
