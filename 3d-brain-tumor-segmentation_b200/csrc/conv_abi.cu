// b3d — C-ABI entry points for the convolution family (see include/b3d.h for the contract).
#include "common.cuh"
#include "conv_common.cuh"

using namespace b3d;

namespace {

struct ConvArgs {
  TView x, w, y;
  int k;
};

// big_halo / small_halo: extra depth slices (slab halos) carried by the respective tensor
int spatial_ok(const TView& big, const TView& small, int stride, const char* what, int big_halo = 0,
               int small_halo = 0) {
  for (int i = 1; i <= 3; ++i) {
    const long long nb = big.shape[i] - (i == 1 ? big_halo : 0), ns = small.shape[i] - (i == 1 ? small_halo : 0);
    if (stride == 1) {
      B3D_REQUIRE(nb == ns, B3D_ERR_SHAPE, "%s: spatial dims differ (dim %d: %lld vs %lld)", what, i, nb, ns);
    } else {
      B3D_REQUIRE(nb % 2 == 0 && nb == 2 * ns, B3D_ERR_SHAPE,
                  "%s: stride-2 needs even sizes with big == 2*small (dim %d: %lld vs %lld)", what, i, nb, ns);
    }
  }
  B3D_REQUIRE(big.shape[0] == small.shape[0], B3D_ERR_SHAPE, "%s: batch differs", what);
  return B3D_OK;
}

int weight_view(const DLTensor* w_, TView* w, int* k) {
  B3D_TRY(view(w_, DT_F32, 5, false, "w", w));
  *k = (int)w->shape[0];
  B3D_REQUIRE((*k == 1 || *k == 3) && w->shape[1] == *k && w->shape[2] == *k, B3D_ERR_UNSUPPORTED,
              "conv: kernel must be 1x1x1 or 3x3x3 (got %lldx%lldx%lld)", (long long)w->shape[0],
              (long long)w->shape[1], (long long)w->shape[2]);
  return B3D_OK;
}

void fill_in(ConvGeom& g, const TView& x) {
  g.B = (int)x.shape[0]; g.Di = (int)x.shape[1]; g.Hi = (int)x.shape[2]; g.Wi = (int)x.shape[3];
  g.Cin = (int)x.shape[4]; g.xp = x.pitch;
}
void fill_out(ConvGeom& g, const TView& y) {
  g.Do = (int)y.shape[1]; g.Ho = (int)y.shape[2]; g.Wo = (int)y.shape[3];
  g.Cout = (int)y.shape[4]; g.yp = y.pitch;
}

int run(const ConvGeom& g, const TView& x, const TView& w, const float* bias, const TView& y,
        const DLTensor* stats_, int groups, const DLTensor* gap_, const DLTensor* wpacked_, cudaStream_t s,
        const TcSources* srcs = nullptr, bool prezeroed = false) {
  // prezeroed: the caller hands in statistics / pooling buffers that are already zero (slices of an arena it clears
  // once per forward) — no memset nodes here
  double* stats = nullptr;
  float* gap = nullptr;
  if (stats_ != nullptr) {
    TView st;
    B3D_TRY(view(stats_, DT_F64, -1, false, "gn_stats", &st));
    const long long S = g.stat_total > 0 ? g.stat_total : (long long)g.Do * g.Ho * g.Wo;
    B3D_REQUIRE(groups >= 1 && g.Cout % groups == 0 && S % groups == 0, B3D_ERR_UNSUPPORTED,
                "conv: fused GN stats need Cout %% groups == 0 and D*H*W %% groups == 0");
    B3D_REQUIRE(st.numel == 2LL * g.B * groups, B3D_ERR_SHAPE, "gn_stats: expected %d fp64 values", 2 * g.B * groups);
    B3D_REQUIRE(y.pitch == g.Cout, B3D_ERR_LAYOUT, "conv: fused GN stats need a contiguous output");
    stats = (double*)st.p;
    if (!prezeroed) B3D_TRY(cuda_ok(cudaMemsetAsync(stats, 0, sizeof(double) * st.numel, s), "memset stats"));
  }
  if (gap_ != nullptr) {
    TView gp;
    B3D_TRY(view(gap_, DT_F32, 2, false, "gap", &gp));
    B3D_REQUIRE(gp.shape[0] == g.B && gp.shape[1] == g.Cout, B3D_ERR_SHAPE, "gap: expected [B, Cout]");
    gap = (float*)gp.p;
    if (!prezeroed) B3D_TRY(cuda_ok(cudaMemsetAsync(gap, 0, sizeof(float) * gp.numel, s), "memset gap"));
  }
  if (wpacked_ != nullptr) {
    TView wp;
    B3D_TRY(view(wpacked_, DT_F32, 1, false, "wpacked", &wp));
    B3D_REQUIRE(tc_conv_supported(g), B3D_ERR_UNSUPPORTED, "conv: shape not supported by the tcgen05 path");
    B3D_REQUIRE((size_t)wp.numel == tc_packed_weight_elems(g), B3D_ERR_SHAPE, "wpacked: wrong size");
    return launch_conv_tc(g, (const float*)x.p, (const float*)wp.p, bias, (float*)y.p, stats, gap, s, srcs);
  }
  B3D_REQUIRE(srcs == nullptr, B3D_ERR_UNSUPPORTED, "conv (P16 operands): only the tcgen05 path (wpacked required)");
  return launch_conv_gather(g, (const float*)x.p, (const float*)w.p, bias, (float*)y.p, stats, gap, s);
}

int bias_ptr(const DLTensor* bias_, int C, const float** out) {
  *out = nullptr;
  if (bias_ == nullptr) return B3D_OK;
  TView b;
  B3D_TRY(view(bias_, DT_F32, 1, false, "bias", &b));
  B3D_REQUIRE(b.numel == C, B3D_ERR_SHAPE, "bias: expected %d values", C);
  *out = (const float*)b.p;
  return B3D_OK;
}

// geometry of forward / dgrad for the four (stride, transposed) variants
int geom_fwd(ConvGeom& g, const TView& x, const TView& w, const TView& y, int k, int stride, int transposed,
             int halo_before = 0, int halo_after = 0) {
  memset(&g, 0, sizeof(g));
  fill_in(g, x);
  fill_out(g, y);
  g.k = k; g.pad = k / 2; g.doff = halo_before;
  const int halo = halo_before + halo_after;
  if (!transposed) {
    B3D_REQUIRE(w.shape[3] == g.Cin && w.shape[4] == g.Cout, B3D_ERR_SHAPE,
                "conv fwd: kernel (..,%lld,%lld) does not match Cin=%d Cout=%d", (long long)w.shape[3],
                (long long)w.shape[4], g.Cin, g.Cout);
    B3D_TRY(spatial_ok(x, y, stride, "conv fwd", halo, 0));
    g.mode = stride == 1 ? CONV_S1 : CONV_DOWN;
    g.wtap = (long long)g.Cin * g.Cout; g.sw_in = g.Cout; g.sw_out = 1;
  } else {
    B3D_REQUIRE(w.shape[3] == g.Cout && w.shape[4] == g.Cin, B3D_ERR_SHAPE,
                "conv-transpose fwd: kernel must be (3,3,3,Cout,Cin)");
    B3D_TRY(spatial_ok(y, x, 2, "conv-transpose fwd", 0, halo));
    g.mode = CONV_UP;
    g.wtap = (long long)g.Cin * g.Cout; g.sw_in = 1; g.sw_out = g.Cin;
  }
  return B3D_OK;
}

int geom_dgrad(ConvGeom& g, const TView& dy, const TView& w, const TView& dx, int k, int stride, int transposed) {
  memset(&g, 0, sizeof(g));
  fill_in(g, dy);   // gathered tensor is dy: "Cin" of the gather = Cout of the layer
  fill_out(g, dx);
  g.k = k; g.pad = k / 2; g.bwd = 1;
  if (!transposed) {
    B3D_REQUIRE(w.shape[3] == g.Cout && w.shape[4] == g.Cin, B3D_ERR_SHAPE, "conv dgrad: kernel/channels mismatch");
    B3D_TRY(spatial_ok(dx, dy, stride, "conv dgrad"));
    g.mode = stride == 1 ? CONV_S1 : CONV_UP;
    g.flip = stride == 1 ? 1 : 0;   // taps reversed
    g.wtap = (long long)g.Cin * g.Cout; g.sw_in = 1; g.sw_out = g.Cin;  // w[t][ci_layer][co_layer]
  } else {
    B3D_REQUIRE(w.shape[3] == g.Cin && w.shape[4] == g.Cout, B3D_ERR_SHAPE, "conv-transpose dgrad: kernel mismatch");
    B3D_TRY(spatial_ok(dy, dx, 2, "conv-transpose dgrad"));
    g.mode = CONV_DOWN;
    g.wtap = (long long)g.Cin * g.Cout; g.sw_in = g.Cout; g.sw_out = 1;  // w[t][co_layer][ci_layer]
  }
  return B3D_OK;
}

}  // namespace

static int conv_fwd_impl(const DLTensor* x_, const DLTensor* w_, const DLTensor* bias_, DLTensor* y_, int stride,
                         int transposed, int act, DLTensor* gn_stats_, int groups, DLTensor* gap_, int accumulate,
                         const DLTensor* wpacked_, int halo_before, int halo_after, void* stream) {
  TView x, w, y;
  int k;
  B3D_TRY(view(x_, DT_F32, 5, true, "x", &x));
  B3D_TRY(view(y_, DT_F32, 5, true, "y", &y));
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_REQUIRE(stride == 1 || (stride == 2 && k == 3), B3D_ERR_UNSUPPORTED, "conv: stride must be 1, or 2 with k=3");
  B3D_REQUIRE(!transposed || stride == 2, B3D_ERR_UNSUPPORTED, "conv-transpose: only k=3 stride=2");
  B3D_REQUIRE(halo_before >= 0 && halo_after >= 0 && halo_before <= 1 && halo_after <= 1 &&
                  (halo_before + halo_after == 0 || x.shape[0] == 1),
              B3D_ERR_ARG, "conv: slab halos are 0 or 1 slice per side, batch 1");
  ConvGeom g;
  B3D_TRY(geom_fwd(g, x, w, y, k, stride, transposed, halo_before, halo_after));
  g.act = act; g.accumulate = accumulate; g.groups = groups;
  const float* bias;
  B3D_TRY(bias_ptr(bias_, g.Cout, &bias));
  return run(g, x, w, bias, y, gn_stats_, groups, gap_, wpacked_, (cudaStream_t)stream);
}

extern "C" int b3d_conv3d_fwd(const DLTensor* x_, const DLTensor* w_, const DLTensor* bias_, DLTensor* y_,
                              int stride, int transposed, int act, DLTensor* gn_stats_, int groups,
                              DLTensor* gap_, int accumulate, const DLTensor* wpacked_, void* stream) {
  return conv_fwd_impl(x_, w_, bias_, y_, stride, transposed, act, gn_stats_, groups, gap_, accumulate, wpacked_, 0, 0,
                       stream);
}

// Depth-slab form for whole-volume inference sharded along D (test.py:133 on a [1,160,192,160,C] volume): x carries
// halo_before / halo_after (0|1) extra depth slices — the neighbour slabs' boundary slices, zeros at the volume
// ends — and y only this slab's slices, so that concatenating the slabs' y equals the conv of the whole volume.
//   conv k3 s1: halos (1,1);  conv k3 s2: (0,1);  conv-transpose: (1,0);  k1: (0,0).
extern "C" int b3d_conv3d_fwd_halo(const DLTensor* x_, const DLTensor* w_, const DLTensor* bias_, DLTensor* y_,
                                   int stride, int transposed, int act, int halo_before, int halo_after,
                                   DLTensor* gap_, const DLTensor* wpacked_, void* stream) {
  return conv_fwd_impl(x_, w_, bias_, y_, stride, transposed, act, nullptr, 1, gap_, 0, wpacked_, halo_before,
                       halo_after, stream);
}

extern "C" int b3d_conv3d_dgrad(const DLTensor* dy_, const DLTensor* w_, DLTensor* dx_, int stride,
                                int transposed, int accumulate, const DLTensor* wpacked_, void* stream) {
  TView dy, w, dx;
  int k;
  B3D_TRY(view(dy_, DT_F32, 5, true, "dy", &dy));
  B3D_TRY(view(dx_, DT_F32, 5, true, "dx", &dx));
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_REQUIRE(stride == 1 || (stride == 2 && k == 3), B3D_ERR_UNSUPPORTED, "conv: stride must be 1, or 2 with k=3");
  ConvGeom g;
  B3D_TRY(geom_dgrad(g, dy, w, dx, k, stride, transposed));
  g.accumulate = accumulate;
  return run(g, dy, w, nullptr, dx, nullptr, 1, nullptr, wpacked_, (cudaStream_t)stream);
}

// TS-mode weight gradient (conv_tc_wgrad_ts.cu) on / off — b3d_set_wgrad_ts, default on
static int g_wgrad_ts = 1;
extern "C" int b3d_set_wgrad_ts(int on) { g_wgrad_ts = on ? 1 : 0; return 0; }

namespace {
// How the tcgen05 weight gradient of a layer is fed: bf16 channels per voxel of the two scratch copies.
//   kind 0: not on the tensor cores (fp32 CUDA-core kernel)
//   kind 1: plain copies (stride 2: the big tensor in space-to-depth order)
//   kind 2: narrow input  (Cin  < 8): x  tap-stacked to pad8(k^3*Cin)  channels, dy plain   (conv_tc_wgrad.cu)
//   kind 3: narrow output (Cout < 8): dy tap-stacked to pad8(k^3*Cout) channels, x  plain
struct WgradPlan { int kind; long long x_ch, dy_ch; };
WgradPlan wgrad_plan(int k, int stride, int transposed, int cin, int cout) {
  WgradPlan p = {0, 0, 0};
  const int taps = k * k * k;
  auto pad8 = [](int v) { return (v + 7) / 8 * 8; };
  if (stride == 1 && !transposed && (k == 1 || k == 3)) {
    if (cin < 8 && cout % 16 == 0 && cout >= 16) { p.kind = 2; p.x_ch = pad8(taps * cin); p.dy_ch = cout; return p; }
    if (cout < 8 && cin % 16 == 0 && cin >= 16) { p.kind = 3; p.x_ch = cin; p.dy_ch = pad8(taps * cout); return p; }
  }
  if (transposed && stride != 2) return p;
  WgradGeom wg;
  memset(&wg, 0, sizeof(wg));
  wg.k = k; wg.s = stride;
  wg.nA = transposed ? cout : cin; wg.nB = transposed ? cin : cout;
  wg.bigp = wg.nA; wg.smallp = wg.nB;
  if (tc_wgrad_supported(wg)) { p.kind = 1; p.x_ch = cin; p.dy_ch = cout; }
  return p;
}
}  // namespace

extern "C" int b3d_conv3d_wgrad(const DLTensor* x_, const DLTensor* dy_, DLTensor* dw_, DLTensor* dbias_,
                                int stride, int transposed, const DLTensor* x_bf16_, const DLTensor* dy_bf16_,
                                int x_bf16_ready, void* stream) {
  TView x, dy, dw;
  int k;
  B3D_TRY(view(x_, DT_F32, 5, true, "x", &x));
  B3D_TRY(view(dy_, DT_F32, 5, true, "dy", &dy));
  B3D_TRY(weight_view(dw_, &dw, &k));
  cudaStream_t s = (cudaStream_t)stream;
  WgradGeom wg;
  memset(&wg, 0, sizeof(wg));
  const TView& big = transposed ? dy : x;
  const TView& sml = transposed ? x : dy;
  B3D_TRY(spatial_ok(big, sml, stride, "conv wgrad"));
  B3D_REQUIRE(dw.shape[3] == big.shape[4] && dw.shape[4] == sml.shape[4], B3D_ERR_SHAPE,
              "conv wgrad: dw channel dims do not match the activations");
  wg.B = (int)big.shape[0];
  wg.Db = (int)big.shape[1]; wg.Hb = (int)big.shape[2]; wg.Wb = (int)big.shape[3]; wg.nA = (int)big.shape[4];
  wg.Ds = (int)sml.shape[1]; wg.Hs = (int)sml.shape[2]; wg.Ws = (int)sml.shape[3]; wg.nB = (int)sml.shape[4];
  wg.k = k; wg.s = stride; wg.pad = stride == 1 ? k / 2 : 0;
  wg.bigp = big.pitch; wg.smallp = sml.pitch;
  float* db = nullptr;
  if (dbias_ != nullptr) {
    TView dbv;
    B3D_TRY(view(dbias_, DT_F32, 1, false, "dbias", &dbv));
    B3D_REQUIRE(dbv.numel == dy.shape[4], B3D_ERR_SHAPE, "dbias: expected %lld values", (long long)dy.shape[4]);
    db = (float*)dbv.p;
  }
  bool bias_done = false;
  if (x_bf16_ != nullptr && dy_bf16_ != nullptr) {
    // tensor-core path: the bf16 scratch copies (caller-allocated, sizes from b3d_conv3d_wgrad_plan) are filled here
    const int cin = (int)x.shape[4], cout = (int)dy.shape[4];
    const WgradPlan pl = wgrad_plan(k, stride, transposed, cin, cout);
    B3D_REQUIRE(pl.kind != 0, B3D_ERR_UNSUPPORTED, "wgrad: shape not on the tcgen05 path");
    TView xb, yb;
    B3D_TRY(view(x_bf16_, DT_BF16, -1, false, "x_bf16", &xb));
    B3D_TRY(view(dy_bf16_, DT_BF16, -1, false, "dy_bf16", &yb));
    const long long nvx = x.numel / cin, nvy = dy.numel / cout;
    B3D_REQUIRE(xb.numel == nvx * pl.x_ch && yb.numel == nvy * pl.dy_ch, B3D_ERR_SHAPE,
                "wgrad: bf16 scratch sizes (expected %lld and %lld elements)", nvx * pl.x_ch, nvy * pl.dy_ch);
    if (pl.kind == 1) {
      B3D_REQUIRE(x.pitch == x.shape[4] && dy.pitch == dy.shape[4], B3D_ERR_LAYOUT, "wgrad (tcgen05): contiguous inputs");
      const TView& bigb = transposed ? yb : xb;
      const TView& smlb = transposed ? xb : yb;
      float* db_big = transposed ? db : nullptr;     // the bias gradient = column sums of dy, whichever role it has
      float* db_sml = transposed ? nullptr : db;
      // x_bf16_ready: the caller already holds the plain bf16 copy of x (two convs of a ResnetBlock share their input)
      const bool skip_big = x_bf16_ready && !transposed && stride == 1, skip_sml = x_bf16_ready && transposed;
      // narrow outputs (Cout <= 32, the 128^3 / 64^3 levels): TS-mode kernel, dy copied in its transposed block order
      const bool ts = g_wgrad_ts && !transposed && stride == 1 && tc_wgrad_ts_supported(wg);
      if (stride == 2)
        B3D_TRY(launch_cast_bf16_s2d((const float*)big.p, bigb.p, wg.B, wg.Ds, wg.Hs, wg.Ws, wg.nA, big.pitch, db_big, s));
      else if (!skip_big)
        B3D_TRY(launch_cast_bf16((const float*)big.p, bigb.p, big.numel / big.shape[4], wg.nA, db_big, s));
      if (ts) {
        B3D_TRY(launch_cast_bf16_t8((const float*)sml.p, smlb.p, sml.numel / sml.shape[4], wg.nB, db_sml, s));
        B3D_TRY(launch_conv_wgrad_ts(wg, bigb.p, smlb.p, (float*)dw.p, s));
      } else {
        if (!skip_sml)
          B3D_TRY(launch_cast_bf16((const float*)sml.p, smlb.p, sml.numel / sml.shape[4], wg.nB, db_sml, s));
        B3D_TRY(launch_conv_wgrad_tc(wg, bigb.p, smlb.p, (float*)dw.p, s));
      }
      bias_done = db != nullptr;
    } else {
      // narrow layer: all taps of the narrow tensor stacked into the M dimension of a single 1x1x1-style GEMM
      const bool nx = pl.kind == 2;
      const TView& nar = nx ? x : dy;       // stacked (narrow) tensor
      const TView& wid = nx ? dy : x;       // plain (wide) tensor
      B3D_REQUIRE(wid.pitch == wid.shape[4], B3D_ERR_LAYOUT, "wgrad (tcgen05): contiguous inputs");
      const int cn = (int)nar.shape[4], nA = (int)(nx ? pl.x_ch : pl.dy_ch);
      B3D_TRY(launch_cast_stack_bf16((const float*)nar.p, (nx ? xb : yb).p, wg.B, wg.Db, wg.Hb, wg.Wb, cn, nar.pitch, k,
                                     nx ? 1 : -1, nA, s));
      B3D_TRY(launch_cast_bf16((const float*)wid.p, (nx ? yb : xb).p, wid.numel / wid.shape[4], (int)wid.shape[4],
                               nx ? db : nullptr, s));
      WgradGeom w1 = wg;
      w1.k = 1; w1.s = 1; w1.pad = 0; w1.nA = nA; w1.nB = (int)wid.shape[4]; w1.bigp = nA; w1.smallp = w1.nB;
      B3D_TRY(launch_conv_wgrad_tc(w1, (nx ? xb : yb).p, (nx ? yb : xb).p, (float*)dw.p, s, k * k * k * cn,
                                   nx ? 0 : cn, dw.numel));
      bias_done = nx && db != nullptr;
    }
  } else {
    B3D_TRY(launch_conv_wgrad(wg, (const float*)big.p, (const float*)sml.p, (float*)dw.p, s));
  }
  if (db != nullptr && !bias_done)
    B3D_TRY(launch_colsum((const float*)dy.p, db, dy.numel / dy.shape[4], (int)dy.shape[4], dy.pitch, true, s));
  return B3D_OK;
}

// bf16 scratch the tcgen05 weight gradient of a layer needs: channels per voxel of the x / dy copies (both 0 when
// the layer's weight gradient runs on the CUDA cores).  Returns the plan kind (see WgradPlan).
extern "C" int b3d_conv3d_wgrad_plan(int k, int stride, int transposed, int cin, int cout, long long* x_ch,
                                     long long* dy_ch) {
  const WgradPlan p = wgrad_plan(k, stride, transposed, cin, cout);
  if (x_ch != nullptr) *x_ch = p.x_ch;
  if (dy_ch != nullptr) *dy_ch = p.dy_ch;
  return p.kind;
}

// 1 when the tcgen05 weight-gradient kernel handles a layer with these LAYER channel counts (k in {1,3} stride 1;
// k3 stride 2 conv / conv-transpose)
extern "C" int b3d_conv3d_wgrad_tc_supported(int k, int stride, int transposed, int cin, int cout) {
  return wgrad_plan(k, stride, transposed, cin, cout).kind != 0 ? 1 : 0;
}

namespace {
// channel roles / weight strides of the gather form for (stride, transposed, dgrad) and kernel dims (.., A, Bc)
void weight_geom(ConvGeom& g, int k, int stride, int transposed, int dgrad, int A, int Bc) {
  memset(&g, 0, sizeof(g));
  g.k = k; g.pad = k / 2; g.bwd = dgrad;
  g.wtap = (long long)A * Bc;
  // contracted channel = A for (conv fwd, convT dgrad), Bc for (conv dgrad, convT fwd)
  const bool contract_a = (transposed != 0) == (dgrad != 0);
  if (contract_a) { g.Cin = A; g.Cout = Bc; g.sw_in = Bc; g.sw_out = 1; }
  else            { g.Cin = Bc; g.Cout = A; g.sw_in = 1; g.sw_out = Bc; }
  if (stride == 1) { g.mode = CONV_S1; g.flip = dgrad; }
  else g.mode = contract_a ? CONV_DOWN : CONV_UP;   // conv s2 fwd & convT dgrad gather DOWN; the other two UP
}
}  // namespace

// 1 when the tcgen05 implicit-GEMM kernel handles this pass of a conv whose Keras kernel is (k,k,k,a,b)
extern "C" int b3d_conv3d_tc_supported(int k, int stride, int transposed, int dgrad, int a, int b) {
  if (!((stride == 1 && !transposed) || (stride == 2 && k == 3))) return 0;
  ConvGeom g;
  weight_geom(g, k, stride, transposed, dgrad, a, b);
  return tc_conv_supported(g) ? 1 : 0;
}

extern "C" long long b3d_conv3d_packed_elems(int k, int stride, int a, int b) {
  ConvGeom g;
  weight_geom(g, k, stride, 0, 0, a, b);
  return (long long)tc_packed_weight_elems(g);
}

// Re-lays a Keras conv kernel out for the tcgen05 kernel, for the forward pass (dgrad=0) or the data gradient
// (dgrad=1) of a Conv3D (transposed=0) / Conv3DTranspose (transposed=1, stride 2) layer.
extern "C" int b3d_conv3d_pack_weights(const DLTensor* w_, DLTensor* packed_, int stride, int transposed, int dgrad,
                                       void* stream) {
  TView w, p;
  int k;
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_TRY(view(packed_, DT_F32, 1, false, "packed", &p));
  B3D_REQUIRE((stride == 1 && !transposed) || (stride == 2 && k == 3), B3D_ERR_UNSUPPORTED,
              "pack_weights: stride 1, or k=3 stride 2 (conv / conv-transpose)");
  ConvGeom g;
  weight_geom(g, k, stride, transposed, dgrad, (int)w.shape[3], (int)w.shape[4]);
  B3D_REQUIRE((size_t)p.numel == tc_packed_weight_elems(g), B3D_ERR_SHAPE, "packed: wrong size");
  return launch_tc_pack_weights(g, (const float*)w.p, (float*)p.p, (cudaStream_t)stream);
}

// Batched form: b3d_conv3d_pack_job writes the table entry of one layer (b3d_conv3d_pack_job_bytes() bytes, host
// memory) and returns the number of 256-thread blocks it needs in *blocks; the caller sets block0 = running sum via
// the `block0` argument, uploads the concatenated entries and calls b3d_conv3d_pack_many once per optimiser step.
extern "C" int b3d_conv3d_pack_job_bytes(void) { return (int)sizeof(PackJob); }

extern "C" int b3d_conv3d_pack_job(const DLTensor* w_, DLTensor* packed_, int stride, int transposed, int dgrad,
                                   long long block0, void* job_out, long long* blocks) {
  TView w, p;
  int k;
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_TRY(view(packed_, DT_F32, 1, false, "packed", &p));
  B3D_REQUIRE(job_out != nullptr && blocks != nullptr, B3D_ERR_ARG, "pack_job: null output");
  B3D_REQUIRE((stride == 1 && !transposed) || (stride == 2 && k == 3), B3D_ERR_UNSUPPORTED,
              "pack_job: stride 1, or k=3 stride 2 (conv / conv-transpose)");
  ConvGeom g;
  weight_geom(g, k, stride, transposed, dgrad, (int)w.shape[3], (int)w.shape[4]);
  B3D_REQUIRE((size_t)p.numel == tc_packed_weight_elems(g), B3D_ERR_SHAPE, "packed: wrong size");
  PackJob jb;
  B3D_TRY(tc_pack_job(g, (const float*)w.p, (float*)p.p, &jb));
  jb.block0 = block0;
  memcpy(job_out, &jb, sizeof(jb));
  *blocks = tc_pack_job_blocks(jb);
  return B3D_OK;
}

extern "C" int b3d_conv3d_pack_many(const DLTensor* jobs_, int njobs, long long blocks, void* stream) {
  TView t;
  static_assert(sizeof(PackJob) % 8 == 0, "PackJob tables travel as int64 tensors");
  B3D_TRY(view(jobs_, DT_I64, 1, false, "jobs", &t));
  B3D_REQUIRE(njobs >= 0 && t.numel * 8 >= (long long)njobs * (long long)sizeof(PackJob), B3D_ERR_SHAPE,
              "pack_many: table too small");
  return launch_tc_pack_many((const PackJob*)t.p, njobs, blocks, (cudaStream_t)stream);
}


// ================================================================================================ P16 operand forms
// The same three passes with the conv INPUT operands given as P16 twins (16-bit [B, D, H, C/8, W, 8], common.cuh) written
// by the producing kernels: no conversion in the loaders (TMA boxes for stride-1 addressing), no cast passes before the
// weight gradient, and channel concatenation (encoder.py:85,91, decoder.py:75) as a list of sources instead of a copy.
namespace {

int p16_sources(const DLTensor* const xs[4], TcSources* src, P16View* first, int* ctot) {
  memset(src, 0, sizeof(*src));
  *ctot = 0;
  for (int i = 0; i < 4; ++i) {
    if (xs[i] == nullptr) break;
    P16View v;
    B3D_TRY(view_p16(xs[i], "x (P16)", &v));
    if (i == 0) *first = v;
    B3D_REQUIRE(v.B == first->B && v.D == first->D && v.H == first->H && v.W == first->W && v.bf16 == first->bf16,
                B3D_ERR_SHAPE, "conv (P16): concatenated sources must agree in batch, space and type");
    src->p[i] = v.p; src->C[i] = 8 * v.C8; src->n = i + 1;
    *ctot += 8 * v.C8;
  }
  B3D_REQUIRE(src->n >= 1, B3D_ERR_ARG, "conv (P16): at least one source");
  src->bf16 = first->bf16;
  return B3D_OK;
}

// a TView standing for the (virtual) NDHWC tensor the P16 sources represent
TView virtual_view(const P16View& v, int C) {
  TView t;
  t.p = v.p; t.ndim = 5;
  t.shape[0] = v.B; t.shape[1] = v.D; t.shape[2] = v.H; t.shape[3] = v.W; t.shape[4] = C;
  t.pitch = C; t.numel = (int64_t)v.B * v.D * v.H * v.W * C;
  return t;
}

}  // namespace

extern "C" int b3d_conv3d_fwd_p16(const DLTensor* x0_, const DLTensor* x1_, const DLTensor* x2_, const DLTensor* x3_,
                                  const DLTensor* w_, const DLTensor* bias_, DLTensor* y_, int stride, int transposed,
                                  int act, DLTensor* gn_stats_, int groups, DLTensor* gap_, int accumulate,
                                  const DLTensor* wpacked_, void* stream) {
  const DLTensor* xs[4] = {x0_, x1_, x2_, x3_};
  TcSources src;
  P16View first;
  int ctot;
  B3D_TRY(p16_sources(xs, &src, &first, &ctot));
  TView w, y;
  int k;
  B3D_TRY(view(y_, DT_F32, 5, true, "y", &y));
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_REQUIRE(stride == 1 || (stride == 2 && k == 3), B3D_ERR_UNSUPPORTED, "conv: stride must be 1, or 2 with k=3");
  B3D_REQUIRE(!transposed || stride == 2, B3D_ERR_UNSUPPORTED, "conv-transpose: only k=3 stride=2");
  B3D_REQUIRE(wpacked_ != nullptr, B3D_ERR_ARG, "conv (P16): packed weights required (tcgen05 path only)");
  const TView x = virtual_view(first, ctot);
  ConvGeom g;
  B3D_TRY(geom_fwd(g, x, w, y, k, stride, transposed));
  g.act = act; g.accumulate = accumulate; g.groups = groups;
  const float* bias;
  B3D_TRY(bias_ptr(bias_, g.Cout, &bias));
  return run(g, x, w, bias, y, gn_stats_, groups, gap_, wpacked_, (cudaStream_t)stream, &src);
}

// The same for one depth slab of a volume (slab.py): the sources carry `halo_before` / `halo_after` extra depth slices
// (the neighbours' boundary slices, received in place), the output holds this slab's slices only, and the fused
// GroupNorm statistics are this slab's PARTIAL sums over the chunks of the whole volume (stat_total output voxels, of
// which this slab's first is stat_off) — the caller all-reduces them.
extern "C" int b3d_conv3d_fwd_p16_slab(const DLTensor* x0_, const DLTensor* x1_, const DLTensor* x2_,
                                       const DLTensor* x3_, const DLTensor* w_, const DLTensor* bias_, DLTensor* y_,
                                       int stride, int transposed, int act, int halo_before, int halo_after,
                                       DLTensor* gn_stats_, int groups, long long stat_off, long long stat_total,
                                       DLTensor* gap_, const DLTensor* wpacked_, int prezeroed, void* stream) {
  const DLTensor* xs[4] = {x0_, x1_, x2_, x3_};
  TcSources src;
  P16View first;
  int ctot;
  B3D_TRY(p16_sources(xs, &src, &first, &ctot));
  TView w, y;
  int k;
  B3D_TRY(view(y_, DT_F32, 5, true, "y", &y));
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_REQUIRE(stride == 1 || (stride == 2 && k == 3), B3D_ERR_UNSUPPORTED, "conv: stride must be 1, or 2 with k=3");
  B3D_REQUIRE(!transposed || stride == 2, B3D_ERR_UNSUPPORTED, "conv-transpose: only k=3 stride=2");
  B3D_REQUIRE(wpacked_ != nullptr, B3D_ERR_ARG, "conv (P16): packed weights required (tcgen05 path only)");
  B3D_REQUIRE(halo_before >= 0 && halo_after >= 0 && halo_before <= 1 && halo_after <= 1 && first.B == 1, B3D_ERR_ARG,
              "conv: slab halos are 0 or 1 slice per side, batch 1");
  const TView x = virtual_view(first, ctot);
  ConvGeom g;
  B3D_TRY(geom_fwd(g, x, w, y, k, stride, transposed, halo_before, halo_after));
  g.act = act; g.groups = groups;
  if (gn_stats_ != nullptr) {
    const long long S = (long long)g.Do * g.Ho * g.Wo;
    B3D_REQUIRE(stat_total > 0 && stat_off >= 0 && stat_off + S <= stat_total, B3D_ERR_ARG,
                "conv (slab): bad statistics window (%lld + %lld of %lld)", stat_off, S, stat_total);
    g.stat_off = stat_off; g.stat_total = stat_total;
  }
  const float* bias;
  B3D_TRY(bias_ptr(bias_, g.Cout, &bias));
  return run(g, x, w, bias, y, gn_stats_, groups, gap_, wpacked_, (cudaStream_t)stream, &src, prezeroed != 0);
}

extern "C" int b3d_conv3d_dgrad_p16(const DLTensor* dy_, const DLTensor* w_, DLTensor* dx_, int stride, int transposed,
                                    int accumulate, const DLTensor* wpacked_, void* stream) {
  const DLTensor* xs[4] = {dy_, nullptr, nullptr, nullptr};
  TcSources src;
  P16View first;
  int ctot;
  B3D_TRY(p16_sources(xs, &src, &first, &ctot));
  TView w, dx;
  int k;
  B3D_TRY(view(dx_, DT_F32, 5, true, "dx", &dx));
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_REQUIRE(stride == 1 || (stride == 2 && k == 3), B3D_ERR_UNSUPPORTED, "conv: stride must be 1, or 2 with k=3");
  B3D_REQUIRE(wpacked_ != nullptr, B3D_ERR_ARG, "conv (P16): packed weights required (tcgen05 path only)");
  const TView dy = virtual_view(first, ctot);
  ConvGeom g;
  B3D_TRY(geom_dgrad(g, dy, w, dx, k, stride, transposed));
  g.accumulate = accumulate;
  return run(g, dy, w, nullptr, dx, nullptr, 1, nullptr, wpacked_, (cudaStream_t)stream, &src);
}

// How the P16 weight gradient of a layer runs: 0 = not on this path (narrow layers, odd channel counts), 1 = straight
// from the operands, 2 = needs a 16-bit scratch of numel(big tensor) elements (stride-2 family: space-to-depth copy),
// 3 = needs a 16-bit scratch of numel(dy) elements (TS-mode kernel: voxel-transposed dy).  `w_sp` = W of dy.
// Data gradient of a stride-1 conv whose INPUT was a virtual channel concat: dx comes out as one compact tensor per
// concatenated piece (dx0 .. dx3, channel counts multiples of 16 adding up to the layer's Cin) instead of one tensor the
// framework would have to slice — and copy — afterwards.
extern "C" int b3d_conv3d_dgrad_p16_split(const DLTensor* dy_, const DLTensor* w_, DLTensor* dx0_, DLTensor* dx1_,
                                          DLTensor* dx2_, DLTensor* dx3_, int accumulate, const DLTensor* wpacked_,
                                          void* stream) {
  const DLTensor* xs[4] = {dy_, nullptr, nullptr, nullptr};
  DLTensor* ds[4] = {dx0_, dx1_, dx2_, dx3_};
  TcSources src;
  P16View first;
  int ctot;
  B3D_TRY(p16_sources(xs, &src, &first, &ctot));
  TView w, d[4];
  int k;
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_REQUIRE(wpacked_ != nullptr, B3D_ERR_ARG, "conv (P16): packed weights required (tcgen05 path only)");
  int n = 0, cin = 0;
  ConvGeom g0;
  memset(&g0, 0, sizeof(g0));
  for (int i = 0; i < 4 && ds[i] != nullptr; ++i, ++n) {
    B3D_TRY(view(ds[i], DT_F32, 5, false, "dx piece", &d[i]));
    B3D_REQUIRE(d[i].shape[4] % 16 == 0 && ((uintptr_t)d[i].p & 31) == 0, B3D_ERR_LAYOUT,
                "dgrad (split): pieces need channels %% 16 == 0 and 32-byte alignment");
    for (int q = 0; q < 4; ++q)
      B3D_REQUIRE(d[i].shape[q] == d[0].shape[q], B3D_ERR_SHAPE, "dgrad (split): pieces differ in batch / space");
    cin += (int)d[i].shape[4];
    g0.yd[i] = (float*)d[i].p; g0.yde[i] = cin;
  }
  B3D_REQUIRE(n >= 1, B3D_ERR_ARG, "dgrad (split): at least one piece");
  TView dx = d[0];                       // the virtual whole: same batch / space, all channels
  dx.shape[4] = cin; dx.pitch = cin; dx.numel = d[0].numel / d[0].shape[4] * cin;
  const TView dy = virtual_view(first, ctot);
  ConvGeom g;
  B3D_TRY(geom_dgrad(g, dy, w, dx, k, 1, 0));
  g.accumulate = accumulate;
  if (n > 1) { g.nyd = n; for (int i = 0; i < n; ++i) { g.yd[i] = g0.yd[i]; g.yde[i] = g0.yde[i]; } }
  return run(g, dy, w, nullptr, dx, nullptr, 1, nullptr, wpacked_, (cudaStream_t)stream, &src);
}

// Data gradient w.r.t. the input of a ResnetBlock from BOTH convs that read it (layers/resnet.py:118,133): the 3x3x3
// conv (gradient dy, kernel w) and the pointwise conv (gradient dres, kernel w_pw) — one kernel: dres joins dy as a
// further K segment that is multiplied with w_pw at the centre tap only.  dx as one compact tensor per piece of a
// virtually concatenated input (one piece: the plain case).
extern "C" int b3d_conv3d_dgrad_p16_block(const DLTensor* dy_, const DLTensor* dres_, const DLTensor* w_,
                                          const DLTensor* wpw_, DLTensor* dx0_, DLTensor* dx1_, DLTensor* dx2_,
                                          DLTensor* dx3_, const DLTensor* wpacked_, const DLTensor* wpacked_pw_,
                                          void* stream) {
  const DLTensor* xs[4] = {dy_, dres_, nullptr, nullptr};
  DLTensor* ds[4] = {dx0_, dx1_, dx2_, dx3_};
  TcSources src;
  P16View first;
  int ctot;
  B3D_TRY(p16_sources(xs, &src, &first, &ctot));
  B3D_REQUIRE(src.n == 2 && src.C[0] == src.C[1], B3D_ERR_SHAPE, "dgrad (block): dy and dres must have the same channels");
  TView w, wpw, d[4], wp, wpc;
  int k, k1;
  B3D_TRY(weight_view(w_, &w, &k));
  B3D_TRY(weight_view(wpw_, &wpw, &k1));
  B3D_REQUIRE(k == 3 && k1 == 1, B3D_ERR_SHAPE, "dgrad (block): a 3x3x3 and a 1x1x1 kernel");
  B3D_REQUIRE(wpacked_ != nullptr && wpacked_pw_ != nullptr, B3D_ERR_ARG, "dgrad (block): packed operands required");
  int n = 0, cin = 0;
  ConvGeom g;
  float* yd[4];
  int yde[4];
  for (int i = 0; i < 4 && ds[i] != nullptr; ++i, ++n) {
    B3D_TRY(view(ds[i], DT_F32, 5, false, "dx piece", &d[i]));
    B3D_REQUIRE(d[i].shape[4] % 16 == 0 && ((uintptr_t)d[i].p & 31) == 0, B3D_ERR_LAYOUT,
                "dgrad (block): pieces need channels %% 16 == 0 and 32-byte alignment");
    for (int q = 0; q < 4; ++q)
      B3D_REQUIRE(d[i].shape[q] == d[0].shape[q], B3D_ERR_SHAPE, "dgrad (block): pieces differ in batch / space");
    cin += (int)d[i].shape[4];
    yd[i] = (float*)d[i].p; yde[i] = cin;
  }
  B3D_REQUIRE(n >= 1, B3D_ERR_ARG, "dgrad (block): at least one piece");
  TView dx = d[0];
  dx.shape[4] = cin; dx.pitch = cin; dx.numel = d[0].numel / d[0].shape[4] * cin;
  const int cb = src.C[0];                               // the block's filters
  const TView dy = virtual_view(first, cb);
  B3D_TRY(geom_dgrad(g, dy, w, dx, 3, 1, 0));            // the 3x3x3 part: checks kernel / channel / spatial agreement
  B3D_REQUIRE(wpw.shape[3] == cin && wpw.shape[4] == cb, B3D_ERR_SHAPE, "dgrad (block): pointwise kernel shape");
  B3D_REQUIRE(tc_conv_supported(g), B3D_ERR_UNSUPPORTED, "dgrad (block): shape not on the tcgen05 path");
  B3D_TRY(view(wpacked_, DT_F32, 1, false, "wpacked", &wp));
  B3D_TRY(view(wpacked_pw_, DT_F32, 1, false, "wpacked (pointwise)", &wpc));
  B3D_REQUIRE((size_t)wp.numel == tc_packed_weight_elems(g), B3D_ERR_SHAPE, "wpacked: wrong size");
  ConvGeom g1 = g;                                       // the pointwise layer's data-gradient geometry (size check)
  g1.k = 1; g1.pad = 0; g1.flip = 0;
  B3D_REQUIRE((size_t)wpc.numel == tc_packed_weight_elems(g1), B3D_ERR_SHAPE, "wpacked (pointwise): wrong size");
  B3D_REQUIRE(tc_operand_type(g) != OP_TF32 && tc_operand_type(g1) == tc_operand_type(g), B3D_ERR_UNSUPPORTED,
              "dgrad (block): 16-bit operands");
  g.Cin = 2 * cb; g.xp = 2 * cb;                          // K = [dy | dres]
  g.c_center = cb; g.wp_center = wpc.p;
  if (n > 1) { g.nyd = n; for (int i = 0; i < n; ++i) { g.yd[i] = yd[i]; g.yde[i] = yde[i]; } }
  return launch_conv_tc(g, (const float*)dy.p, (const float*)wp.p, nullptr, (float*)dx.p, nullptr, nullptr,
                        (cudaStream_t)stream, &src);
}

extern "C" int b3d_conv3d_wgrad_p16_plan(int k, int stride, int transposed, int cin, int cout, int w_sp) {
  const WgradPlan p = wgrad_plan(k, stride, transposed, cin, cout);
  if (p.kind != 1 || cin % 8 != 0 || cout % 8 != 0) return 0;
  if (stride == 2) return 2;
  WgradGeom wg;
  memset(&wg, 0, sizeof(wg));
  wg.k = k; wg.s = 1; wg.nA = cin; wg.nB = cout; wg.bigp = cin; wg.smallp = cout; wg.Ws = w_sp;
  return (g_wgrad_ts && tc_wgrad_ts_supported(wg)) ? 3 : 1;
}

// Both weight gradients of a ResnetBlock's input convs in one pass over x (resnet.py:118 pointwise, :133 first 3x3x3):
// dw = the 3x3x3 layer's (x, dy), dw_pw = the pointwise layer's (x, dres).  kd-in-M kernel only (stride 1, Cin = 16 or a
// multiple of 32 up to 128, Cout 16 | 32, W % 8 == 0, H % 2 == 0): b3d_conv3d_wgrad_p16_block_ok tells.
extern "C" int b3d_conv3d_wgrad_p16_block_ok(int cin, int cout, int h_sp, int w_sp) {
  WgradGeom wg;
  memset(&wg, 0, sizeof(wg));
  wg.k = 3; wg.s = 1; wg.nA = cin; wg.nB = cout; wg.Ws = w_sp; wg.Hs = h_sp;
  WgP16 wp;
  memset(&wp, 0, sizeof(wp));
  wp.n = 1; wp.C[0] = cin; wp.big_bf16 = wp.small_bf16 = 1;
  return tc_wgrad_kdf_supported(wg, &wp) ? 1 : 0;
}

extern "C" int b3d_conv3d_wgrad_p16_block(const DLTensor* x0_, const DLTensor* x1_, const DLTensor* x2_,
                                          const DLTensor* x3_, const DLTensor* dy_, const DLTensor* dres_, DLTensor* dw_,
                                          DLTensor* dw_pw_, void* stream) {
  const DLTensor* xs[4] = {x0_, x1_, x2_, x3_};
  TcSources src;
  P16View xf, dy, dres;
  int cin;
  B3D_TRY(p16_sources(xs, &src, &xf, &cin));
  B3D_TRY(view_p16(dy_, "dy (P16)", &dy));
  B3D_TRY(view_p16(dres_, "dres (P16)", &dres));
  TView dw, dwp;
  int k, kp;
  B3D_TRY(weight_view(dw_, &dw, &k));
  B3D_TRY(weight_view(dw_pw_, &dwp, &kp));
  const int cout = 8 * dy.C8;
  B3D_REQUIRE(k == 3 && kp == 1, B3D_ERR_SHAPE, "wgrad (block): a 3x3x3 and a 1x1x1 kernel");
  B3D_REQUIRE(xf.bf16 && dy.bf16 && dres.bf16, B3D_ERR_DTYPE, "wgrad (block): bf16 twins of all operands");
  B3D_REQUIRE(dres.B == dy.B && dres.D == dy.D && dres.H == dy.H && dres.W == dy.W && dres.C8 == dy.C8, B3D_ERR_SHAPE,
              "wgrad (block): dres must match dy");
  B3D_REQUIRE(xf.B == dy.B && xf.D == dy.D && xf.H == dy.H && xf.W == dy.W, B3D_ERR_SHAPE, "wgrad (block): spatial dims");
  B3D_REQUIRE(dw.shape[3] == cin && dw.shape[4] == cout && dwp.shape[3] == cin && dwp.shape[4] == cout, B3D_ERR_SHAPE,
              "wgrad (block): dw channel dims");
  WgradGeom wg;
  memset(&wg, 0, sizeof(wg));
  wg.B = xf.B; wg.Db = xf.D; wg.Hb = xf.H; wg.Wb = xf.W; wg.nA = cin;
  wg.Ds = dy.D; wg.Hs = dy.H; wg.Ws = dy.W; wg.nB = cout;
  wg.k = 3; wg.s = 1; wg.pad = 1;
  wg.bigp = cin; wg.smallp = cout;
  WgP16 wp;
  memset(&wp, 0, sizeof(wp));
  wp.small = dy.p; wp.small_bf16 = 1; wp.big_bf16 = 1;
  wp.n = src.n;
  for (int i = 0; i < src.n; ++i) { wp.big[i] = src.p[i]; wp.C[i] = src.C[i]; }
  B3D_REQUIRE(tc_wgrad_kdf_supported(wg, &wp), B3D_ERR_UNSUPPORTED, "wgrad (block): layer not on the kd-in-M path (%d->%d)",
              cin, cout);
  return launch_conv_wgrad_kdf(wg, (float*)dw.p, (cudaStream_t)stream, wp, dres.p, (float*)dwp.p);
}

extern "C" int b3d_conv3d_wgrad_narrow_ok(int k, int cin, int cout, int pair) {
  return tc_wgrad_narrow_supported(k, cin, cout, pair) ? 1 : 0;
}

extern "C" int b3d_conv3d_wgrad_narrow(const DLTensor* nar_, const DLTensor* wide_, const DLTensor* wide2_, DLTensor* dw_,
                                       DLTensor* dw2_, DLTensor* dbias_, void* stream) {
  TView nar, dw;
  P16View wide;
  int k;
  B3D_TRY(view(nar_, DT_F32, 5, true, "narrow tensor", &nar));
  B3D_TRY(view_p16(wide_, "wide tensor (P16)", &wide));
  B3D_TRY(weight_view(dw_, &dw, &k));
  B3D_REQUIRE(wide.bf16, B3D_ERR_DTYPE, "wgrad (narrow): the wide operand is a bf16 twin");
  NarrowWgrad a;
  memset(&a, 0, sizeof(a));
  a.nar = (const float*)nar.p; a.pitch = nar.pitch;
  a.B = (int)nar.shape[0]; a.D = (int)nar.shape[1]; a.H = (int)nar.shape[2]; a.W = (int)nar.shape[3];
  a.Cn = (int)nar.shape[4]; a.k = k; a.Cw = 8 * wide.C8;
  a.wide = wide.p; a.dw = (float*)dw.p;
  B3D_REQUIRE(wide.B == a.B && wide.D == a.D && wide.H == a.H && wide.W == a.W, B3D_ERR_SHAPE,
              "wgrad (narrow): spatial dims of the two operands differ");
  if (dw.shape[3] == a.Cn && dw.shape[4] == a.Cw) a.tr = 0;
  else if (dw.shape[3] == a.Cw && dw.shape[4] == a.Cn) a.tr = 1;
  else B3D_REQUIRE(false, B3D_ERR_SHAPE, "wgrad (narrow): dw channel dims match neither operand order");
  if (wide2_ != nullptr || dw2_ != nullptr) {
    P16View w2;
    TView dw2;
    int k2;
    B3D_REQUIRE(wide2_ != nullptr && dw2_ != nullptr && a.tr == 0, B3D_ERR_ARG,
                "wgrad (narrow): dres and dw_pw go together, with a narrow layer input");
    B3D_TRY(view_p16(wide2_, "dres (P16)", &w2));
    B3D_TRY(weight_view(dw2_, &dw2, &k2));
    B3D_REQUIRE(w2.bf16 && w2.B == wide.B && w2.D == wide.D && w2.H == wide.H && w2.W == wide.W && w2.C8 == wide.C8,
                B3D_ERR_SHAPE, "wgrad (narrow): dres must match dy");
    B3D_REQUIRE(k2 == 1 && dw2.shape[3] == a.Cn && dw2.shape[4] == a.Cw, B3D_ERR_SHAPE,
                "wgrad (narrow): dw_pw is the (1,1,1,Cin,Cout) kernel gradient");
    a.wide2 = w2.p; a.dw2 = (float*)dw2.p;
  }
  if (dbias_ != nullptr) {
    TView db;
    B3D_TRY(view(dbias_, DT_F32, 1, false, "dbias", &db));
    B3D_REQUIRE(a.tr == 1 && db.numel == a.Cn, B3D_ERR_ARG,
                "wgrad (narrow): the bias gradient is the column sums of a narrow dy (%d values)", a.Cn);
    a.dbias = (float*)db.p;
  }
  return launch_conv_wgrad_narrow(a, (cudaStream_t)stream);
}

// dw of a Conv3D (x = layer input, up to 4 concatenated P16 sources; dy = P16 gradient of the output) or of a
// Conv3DTranspose (transposed = 1: single source).  The bias gradient is NOT produced here: on this path it is emitted
// by the kernel that writes dy (b3d_gn_bwd_apply / b3d_block_epilogue_bwd_apply, `dbias`).
extern "C" int b3d_conv3d_wgrad_p16(const DLTensor* x0_, const DLTensor* x1_, const DLTensor* x2_, const DLTensor* x3_,
                                    const DLTensor* dy_, DLTensor* dw_, int stride, int transposed, DLTensor* scratch_,
                                    void* stream) {
  const DLTensor* xs[4] = {x0_, x1_, x2_, x3_};
  TcSources src;
  P16View xf, dy;
  int cin;
  B3D_TRY(p16_sources(xs, &src, &xf, &cin));
  B3D_TRY(view_p16(dy_, "dy (P16)", &dy));
  TView dw;
  int k;
  B3D_TRY(weight_view(dw_, &dw, &k));
  cudaStream_t s = (cudaStream_t)stream;
  const int cout = 8 * dy.C8;
  B3D_REQUIRE(!transposed || src.n == 1, B3D_ERR_UNSUPPORTED, "wgrad (P16): conv-transpose takes one source");
  B3D_REQUIRE(xf.bf16 && dy.bf16, B3D_ERR_DTYPE,
              "wgrad (P16): bf16 twins of both operands (kind::f16 takes one operand type; forward activations carry a "
              "second, bf16 twin for this pass)");
  const int plan = b3d_conv3d_wgrad_p16_plan(k, stride, transposed, cin, cout, dy.W);
  B3D_REQUIRE(plan != 0, B3D_ERR_UNSUPPORTED, "wgrad (P16): layer not on this path (k=%d s=%d %d->%d)", k, stride, cin, cout);
  const P16View& big = transposed ? dy : xf;
  const P16View& sml = transposed ? xf : dy;
  const int cbig = transposed ? cout : cin, csml = transposed ? cin : cout;
  B3D_REQUIRE(dw.shape[3] == cbig && dw.shape[4] == csml, B3D_ERR_SHAPE, "wgrad (P16): dw channel dims");
  B3D_REQUIRE(big.B == sml.B && big.D == stride * sml.D && big.H == stride * sml.H && big.W == stride * sml.W,
              B3D_ERR_SHAPE, "wgrad (P16): spatial dims");
  WgradGeom wg;
  memset(&wg, 0, sizeof(wg));
  wg.B = big.B; wg.Db = big.D; wg.Hb = big.H; wg.Wb = big.W; wg.nA = cbig;
  wg.Ds = sml.D; wg.Hs = sml.H; wg.Ws = sml.W; wg.nB = csml;
  wg.k = k; wg.s = stride; wg.pad = stride == 1 ? k / 2 : 0;
  wg.bigp = cbig; wg.smallp = csml;
  void* scratch = nullptr;
  long long scratch_n = 0;
  if (scratch_ != nullptr) {
    TView sc;
    B3D_TRY(view(scratch_, scratch_->dtype.code == kDLBfloat ? DT_BF16 : DT_F16, -1, false, "scratch", &sc));
    scratch = sc.p; scratch_n = sc.numel;
    B3D_REQUIRE(((uintptr_t)scratch & 15) == 0, B3D_ERR_LAYOUT, "scratch: alignment");
  }
  WgP16 wp;
  memset(&wp, 0, sizeof(wp));
  wp.small = sml.p; wp.small_bf16 = sml.bf16; wp.big_bf16 = big.bf16;
  if (plan == 2) {
    const long long need = (long long)big.B * big.D * big.H * big.W * cbig;
    B3D_REQUIRE(scratch != nullptr && scratch_n >= need, B3D_ERR_ARG, "wgrad (P16, stride 2): scratch of %lld elements", need);
    int c8off = 0;
    const int c8tot = cbig / 8;
    if (transposed) {
      B3D_TRY(launch_p16_s2d(big.p, scratch, big.B, sml.D, sml.H, sml.W, big.C8, 0, c8tot, s));
    } else {
      for (int i = 0; i < src.n; ++i) {
        B3D_TRY(launch_p16_s2d(src.p[i], scratch, big.B, sml.D, sml.H, sml.W, src.C[i] / 8, c8off, c8tot, s));
        c8off += src.C[i] / 8;
      }
    }
    wp.n = 1; wp.big[0] = scratch; wp.C[0] = 8 * cbig;
    return launch_conv_wgrad_tc(wg, scratch, sml.p, (float*)dw.p, s, 0, 0, 0, &wp);
  }
  if (!transposed) {
    wp.n = src.n;
    for (int i = 0; i < src.n; ++i) { wp.big[i] = src.p[i]; wp.C[i] = src.C[i]; }
    // depth taps folded into M (Cin = 32, and Cin = 16 ahead of the TS-mode kernel of plan 3)
    if (tc_wgrad_kdf_supported(wg, &wp)) return launch_conv_wgrad_kdf(wg, (float*)dw.p, s, wp);
  }
  if (plan == 3) {
    const long long need = (long long)dy.B * dy.D * dy.H * dy.W * cout;
    B3D_REQUIRE(scratch != nullptr && scratch_n >= need, B3D_ERR_ARG, "wgrad (P16, TS): scratch of %lld elements", need);
    if (src.n == 1 && g_wgrad_ts && tc_wgrad_ts_supported(wg)) {
      B3D_TRY(launch_p16_t8(dy.p, scratch, (long long)dy.B * dy.D * dy.H, dy.W, dy.C8, s));
      return launch_conv_wgrad_ts(wg, xf.p, scratch, (float*)dw.p, s, 1, 0);
    }
    // the TS kernel takes one source only: the plan-1 kernel below (the scratch stays unused)
  }
  if (transposed) { wp.n = 1; wp.big[0] = big.p; wp.C[0] = cbig; }
  return launch_conv_wgrad_tc(wg, big.p, sml.p, (float*)dw.p, s, 0, 0, 0, &wp);
}
