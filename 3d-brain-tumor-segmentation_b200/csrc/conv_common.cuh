// b3d — geometry descriptors shared by the generic and tcgen05 convolution paths.
#pragma once
#include <cuda_runtime.h>

namespace b3d {

enum { CONV_S1 = 0, CONV_DOWN = 1, CONV_UP = 2 };
enum { OP_TF32 = 0, OP_BF16 = 1, OP_F16 = 2 };   // operand type of the tcgen05 conv MMAs

// gather form:  y[b,o,co] = act( sum_{t,ci} x[b,pos(o,t),ci] * w[tw(t)*wtap + ci*sw_in + co*sw_out] + bias[co] )
struct ConvGeom {
  int B, Di, Hi, Wi, Cin;   // input  (gathered) tensor
  int Do, Ho, Wo, Cout;     // output tensor
  int k, pad, mode, flip;   // kernel size (1|3), S1 padding, CONV_*, reverse taps
  long long xp, yp;         // channel pitch of x / y (elements per voxel row)
  long long wtap;           // elements between taps in w (= A*B)
  int sw_in, sw_out;        // strides of the contracted / produced channel in w
  int act, accumulate;      // 1 = sigmoid; y += result
  int groups;               // GN groups when stats are requested
  int bwd;                  // 1 = backward pass (operand-precision choice of the tcgen05 path)
  int doff;                 // slab halos: logical input depth slice i lives at buffer slice i + doff (of Di)
  // depth-slab inference with fused GroupNorm statistics: the output tensor is voxels [stat_off, stat_off + Do*Ho*Wo) of
  // a volume of stat_total voxels whose 1/groups chunks the statistics are taken over (0 / 0: the tensor is the volume)
  long long stat_off, stat_total;
  // output split by channel ranges into separate compact tensors (the data gradient of a conv whose input is a virtual
  // concat: one tensor per concatenated piece, no slicing copies afterwards).  nyd = 0: one output (y, yp).
  // 3x3x3 stride-1 only: the last c_center input channels are multiplied with the packed 1x1x1 operand wp_center at the
  // centre tap only (conv_tc.cu, TcParams::cfull); Cin counts them, the 3x3x3 packed operand does not
  int c_center;
  const void* wp_center;
  int nyd;
  float* yd[4];
  int yde[4];               // cumulative channel end of piece i (multiples of 16)
};

// outer-product form:  dw[t][a][b] = sum_{n,o} big[n, s*o+t-pad, a] * small[n, o, b]
struct WgradGeom {
  int B, Db, Hb, Wb, nA;    // "big" tensor (the one indexed with the tap offset)
  int Ds, Hs, Ws, nB;       // "small" tensor
  int k, s, pad;
  long long bigp, smallp;   // channel pitches
};

int launch_conv_gather(const ConvGeom& cg, const float* x, const float* w, const float* bias, float* y,
                       double* stats, float* gap, cudaStream_t s);
int launch_conv_wgrad(const WgradGeom& wg, const float* big, const float* small, float* dw, cudaStream_t s);
int launch_colsum(const float* x, float* out, long long N, int C, long long pitch, bool zero, cudaStream_t s);

// tcgen05 path (conv_tc.cu).  Returns true when the shape is handled there.
bool tc_conv_supported(const ConvGeom& cg);
// P16 input operand of the tcgen05 conv: up to 4 source tensors [B, Di, Hi, C_i/8, Wi, 8] (16-bit) whose channels are
// concatenated virtually (encoder.py:85,91 / decoder.py:75 without a copy); all fp16 (forward) or all bf16 (backward)
struct TcSources {
  int n;
  const void* p[4];
  int C[4];
  int bf16;
};
int launch_conv_tc(const ConvGeom& cg, const float* x, const float* wpacked, const float* bias, float* y,
                   double* stats, float* gap, cudaStream_t s, const TcSources* srcs = nullptr);
size_t tc_packed_weight_elems(const ConvGeom& cg);
int launch_pack_s2(const ConvGeom& cg, const float* w, float* wpacked, int op, cudaStream_t s);
int launch_tc_pack_weights(const ConvGeom& cg, const float* w, float* wpacked, cudaStream_t s);

// one layer's operand re-layout as a table entry of pack_many_kernel (conv_tc.cu): all layers in one launch
struct PackJob {
  const float* w;           // Keras-layout weights
  void* wp;                 // packed operand
  long long total;          // packed elements
  long long block0;         // first block of this job in the batched grid
  long long wtap;
  int s2, op, up, taps;     // stride-2 family?, OP_*, UP-type (s2), taps (S1)
  int Cin, Cout, N;         // S1: padded channel counts, N tile;  s2: real Cg, Cp, N tile
  int sw_in, sw_out;
  int aux;                  // S1: flip;  s2: NTdown
  int cin_real, cout_real;  // S1 zero-padding bounds
};
int tc_pack_job(const ConvGeom& cg, const float* w, float* wpacked, PackJob* job);
long long tc_pack_job_blocks(const PackJob& job);
int launch_tc_pack_many(const PackJob* jobs_dev, int njobs, long long blocks, cudaStream_t s);

#ifdef __CUDACC__
// element i of the packed 2x2x2 stride-1 operand of a DOWN / UP geometry (layout and index algebra: conv_s2.cu)
__device__ __forceinline__ float pack_s2_elem(const float* __restrict__ w, long long i, int T, int up, int Cg, int Cp,
                                              int N, long long wtap, int sw_in, int sw_out, int NTdown) {
  const int K = up ? Cg : 8 * Cg;
  const int nch = K / (2 * T);
  long long r = i;
  const int j = (int)(r % T); r /= T;
  const int n = (int)(r % N); r /= N;
  const int pl = (int)(r % 2); r /= 2;
  const int tap = (int)(r % 8); r /= 8;
  const int c = (int)(r % nch); r /= nch;
  const int ns = (int)r;
  const int k = 2 * T * c + T * pl + j, nn = ns * N + n;
  int p, cg, cp;
  if (up) { cg = k; p = nn / Cp; cp = nn % Cp; }
  else    { p = k / Cg; cg = k % Cg; cp = nn; }
  const int kd = tap >> 2, kh = (tap >> 1) & 1, kw = tap & 1;
  const int pd = p >> 2, ph = (p >> 1) & 1, pw = p & 1;
  const int td = up ? pd + 2 * (1 - kd) : 2 * kd + pd;
  const int th = up ? ph + 2 * (1 - kh) : 2 * kh + ph;
  const int tw = up ? pw + 2 * (1 - kw) : 2 * kw + pw;
  (void)NTdown;
  if (td <= 2 && th <= 2 && tw <= 2 && cp < Cp)
    return w[(long long)((td * 3 + th) * 3 + tw) * wtap + (long long)cg * sw_in + (long long)cp * sw_out];
  return 0.f;
}
#endif

int tc_operand_type(const ConvGeom& g);   // OP_* the tcgen05 conv will use for this geometry / pass
int tc_pick_n(int Cout);               // N tile of the tcgen05 conv for this output-channel count

bool tc_wgrad_supported(const WgradGeom& wg);
// P16 operands of the weight gradient: `big` = up to 4 sources concatenating to the big tensor's channels (for the
// stride-2 family: ONE coarse space-to-depth tensor, launch_p16_s2d), `small` = one tensor
struct WgP16 {
  int n;
  const void* big[4];
  int C[4];
  int big_bf16;
  const void* small;
  int small_bf16;
};
int launch_conv_wgrad_tc(const WgradGeom& wg, const void* x_bf16, const void* dy_bf16, float* dw, cudaStream_t s,
                         int rows_real = 0, int tr_cn = 0, long long dw_elems = 0, const WgP16* p16 = nullptr);
int launch_p16_s2d(const void* src, void* dst, int B, int D, int H, int W, int C8, int c8off, int C8tot, cudaStream_t s);
int launch_p16_t8(const void* src, void* dst, long long rows, int W, int C8, cudaStream_t s);
// TS-mode weight gradient for narrow outputs (conv_tc_wgrad_ts.cu)
bool tc_wgrad_ts_supported(const WgradGeom& wg);
int launch_conv_wgrad_ts(const WgradGeom& wg, const void* x_bf16, const void* dyT_bf16, float* dw, cudaStream_t s,
                         int x_p16 = 0, int x_f16 = 0);
// 3x3x3 weight gradient with the depth taps folded into M (conv_tc_wgrad.cu): Cin 32 | 64, Cout 16 | 32, P16 sources
bool tc_wgrad_kdf_supported(const WgradGeom& wg, const WgP16* p16);
int launch_conv_wgrad_kdf(const WgradGeom& wg, float* dw, cudaStream_t s, const WgP16& p16,
                          const void* dres = nullptr, float* dw2 = nullptr);
// weight gradient of a stride-1 k in {1, 3} layer with Cn < 8 channels on one side, the tap-stacked operand of the
// narrow fp32 tensor built in shared memory (conv_tc_wgrad.cu); the wide side is a bf16 P16 twin
struct NarrowWgrad {
  const float* nar;                // fp32 [B, D, H, W, pitch], Cn channels
  long long pitch;
  int B, D, H, W, Cn, k;
  int tr;                          // 0: nar = layer input x, dw [k,k,k,Cn,Cw]; 1: nar = dy, dw [k,k,k,Cw,Cn]
  const void* wide;                // P16 bf16 twin, Cw channels: dy (tr = 0) or x (tr = 1)
  const void* wide2;               // nullable (tr = 0): dres of the pointwise conv reading the same x
  int Cw;
  float* dw;
  float* dw2;                      // with wide2: the pointwise conv's dw [Cn][Cw]
  float* dbias;                    // nullable (tr = 1): column sums of dy
};
bool tc_wgrad_narrow_supported(int k, int cin, int cout, int pair);
int launch_conv_wgrad_narrow(const NarrowWgrad& a, cudaStream_t s);
int launch_cast_bf16_t8(const float* src, void* dst, long long nvox, int C, float* colsum, cudaStream_t s);
int launch_cast_stack_bf16(const float* src, void* dst, int B, int D, int H, int W, int Cn, long long pitch, int k,
                           int sgn, int nA, cudaStream_t s);
int launch_cast_bf16(const float* src, void* dst, long long nvox, int C, float* colsum, cudaStream_t s);
int launch_cast_bf16_s2d(const float* src, void* dst, int B, int D, int H, int W, int C, long long pitch,
                         float* colsum, cudaStream_t s);

}  // namespace b3d
