// b3d — error channel + DLPack validation shared by every C-ABI entry point.
#include <stdarg.h>

#include "common.cuh"

namespace b3d {

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int view(const DLTensor* t, int dtype, int ndim, bool allow_pitch, const char* name, TView* out) {
  B3D_REQUIRE(t != nullptr, B3D_ERR_ARG, "%s: null tensor", name);
  B3D_REQUIRE(t->device.device_type == kDLCUDA, B3D_ERR_DEVICE,
              "%s: tensor must live on a CUDA device (device_type=%d); b3d has no CPU path", name,
              (int)t->device.device_type);
  static const struct { uint8_t code, bits; } kDT[] = {
      {kDLFloat, 32}, {kDLFloat, 64}, {kDLInt, 64}, {kDLBfloat, 16}, {kDLFloat, 16}, {kDLUInt, 8}};
  B3D_REQUIRE(t->dtype.code == kDT[dtype].code && t->dtype.bits == kDT[dtype].bits && t->dtype.lanes == 1,
              B3D_ERR_DTYPE, "%s: wrong dtype (code=%d bits=%d), expected code=%d bits=%d", name,
              (int)t->dtype.code, (int)t->dtype.bits, (int)kDT[dtype].code, (int)kDT[dtype].bits);
  B3D_REQUIRE(ndim < 0 || t->ndim == ndim, B3D_ERR_SHAPE, "%s: ndim=%d, expected %d", name, t->ndim, ndim);
  B3D_REQUIRE(t->ndim >= 1 && t->ndim <= 6, B3D_ERR_SHAPE, "%s: ndim=%d unsupported", name, t->ndim);
  out->ndim = t->ndim;
  out->device = t->device.device_id;
  int64_t n = 1;
  for (int i = 0; i < t->ndim; ++i) {
    out->shape[i] = t->shape[i];
    n *= t->shape[i];
  }
  out->numel = n;
  const int last = t->ndim - 1;
  out->pitch = t->shape[last];
  if (t->strides != nullptr && n > 0) {
    // tolerate arbitrary strides on size-1 dims
    int64_t pitch = t->shape[last];
    if (t->shape[last] != 1)
      B3D_REQUIRE(t->strides[last] == 1, B3D_ERR_LAYOUT, "%s: innermost stride must be 1 (NDHWC compact)", name);
    if (last >= 1) {
      // find the pitch from the first non-unit outer dim
      for (int i = last - 1; i >= 0; --i) {
        if (t->shape[i] != 1) {
          int64_t inner = 1;
          for (int j = i + 1; j < last; ++j) inner *= t->shape[j];
          B3D_REQUIRE(t->strides[i] % inner == 0, B3D_ERR_LAYOUT, "%s: non-compact strides", name);
          pitch = t->strides[i] / inner;
          break;
        }
      }
      B3D_REQUIRE(pitch >= t->shape[last], B3D_ERR_LAYOUT, "%s: overlapping strides", name);
      int64_t expect = pitch;
      for (int i = last - 1; i >= 0; --i) {
        if (t->shape[i] != 1)
          B3D_REQUIRE(t->strides[i] == expect, B3D_ERR_LAYOUT,
                      "%s: strides are not compact NDHWC (dim %d stride %lld, expected %lld)", name, i,
                      (long long)t->strides[i], (long long)expect);
        expect *= t->shape[i];
      }
    }
    B3D_REQUIRE(allow_pitch || pitch == t->shape[last], B3D_ERR_LAYOUT,
                "%s: must be contiguous (channel-sliced views not accepted here)", name);
    out->pitch = pitch;
  }
  out->p = (char*)t->data + t->byte_offset;
  return B3D_OK;
}

int view_p16(const DLTensor* t, const char* name, P16View* out) {
  B3D_REQUIRE(t != nullptr, B3D_ERR_ARG, "%s: null tensor", name);
  B3D_REQUIRE(t->dtype.bits == 16 && t->dtype.lanes == 1 && (t->dtype.code == kDLBfloat || t->dtype.code == kDLFloat),
              B3D_ERR_DTYPE, "%s: P16 operands are fp16 or bf16", name);
  TView v;
  B3D_TRY(view(t, t->dtype.code == kDLBfloat ? DT_BF16 : DT_F16, 6, false, name, &v));
  B3D_REQUIRE(v.shape[5] == 8, B3D_ERR_LAYOUT, "%s: P16 layout is [B, D, H, C/8, W, 8]", name);
  B3D_REQUIRE(((uintptr_t)v.p & 15) == 0, B3D_ERR_LAYOUT, "%s: P16 operands must be 16-byte aligned", name);
  out->p = v.p;
  out->B = (int)v.shape[0]; out->D = (int)v.shape[1]; out->H = (int)v.shape[2]; out->C8 = (int)v.shape[3];
  out->W = (int)v.shape[4];
  out->bf16 = t->dtype.code == kDLBfloat ? 1 : 0;
  return B3D_OK;
}

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

}  // namespace b3d

extern "C" const char* b3d_last_error(void) { return b3d::g_err; }
extern "C" int b3d_abi_version(void) { return 2; }
